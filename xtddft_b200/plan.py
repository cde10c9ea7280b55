"""Sigma-build plans: each method of the spin-adapted TDA family compiled to generic descriptors.

The CUDA engine (`csrc/`) knows nothing about X-TDA / SF-TDA / XSF-TDA.  It executes a *plan*:

  channels     z blocks [occ x vir] with their MO index lists (zero "pad" orbitals keep every block start
               on an even column, which the TMA loads need)
  k_terms      MO-resident exchange  sigma[i,a] += sum_P sum_jb w(iblk,ablk,jblk,bblk) L^P_ij z_jb L^P_ba
               (one build covers hyb*K of A and every K image of Delta A through the block weights)
  j_blocks     Coulomb images on (sub-)blocks: rho^P_src = <L^P_blk, z_blk>,  sigma_blk += sum_P (mix rho)^P L^P_blk
  xc           grid kernel kind (UKS f_xc, spin-flip ALDA0, multicollinear)
  local terms  Fock and Delta-A Fock-like couplings as small right / left GEMMs, rank-1 trace terms, diagonals
  layout       sparse maps between the caller's vector layout and the engine's padded block layout

This file turns the reference's formulas into those descriptors:
  X-TDA   xtddft/XTDA.py:558-692           (SURVEY Appendix A.1)
  SF-TDA  xtddft/SF_TDA.py:162-286         (Appendix A.2)
  XSF-TDA xtddft/XSF_TDA.py:915-1290, xtddft/XSF_TDA_GPU.py:357-729 (Appendix A.3, A.5)
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import List, Optional, Tuple

import numpy as np

from .problem import ProblemData

# layouts accepted at the vind boundary (SURVEY Appendix A.5)
LAYOUT_PYSCF = "pyscf"       # PySCF vector order
LAYOUT_BLOCK = "block"       # cv | co | ov | oo  (XSF_TDA CPU class)


def _even(n: int) -> int:
    return n + (n & 1)


@dataclass
class ChannelSpec:
    spin_o: int
    occ_idx: np.ndarray            # int32 MO column per internal occ position, -1 = zero pad
    spin_v: int
    vir_idx: np.ndarray
    o_blocks: List[Tuple[int, int]]  # (start, n) of each occ block in internal positions
    v_blocks: List[Tuple[int, int]]

    @property
    def no(self) -> int:
        return len(self.occ_idx)

    @property
    def nv(self) -> int:
        return len(self.vir_idx)


@dataclass
class KTerm:
    tensor: int                    # 0: full-range cderi, 1: long-range cderi
    ch: int
    weights: np.ndarray            # [n_oblk, n_vblk, n_oblk, n_vblk]  (iblk, ablk, jblk, bblk)


@dataclass
class KTermT:
    """Exchange of the transposed trial density: sigma[i,a] += weight * sum_P sum_jb L^P_ib z_jb L^P_ja (Z-vector plans)."""
    tensor: int
    ch: int
    weight: float


@dataclass
class JBlock:
    ch: int
    r0: int
    nr: int
    c0: int
    nc: int


@dataclass
class LocalGemm:
    side: str                      # 'R': dst[r,c] += a * sum_b src[r,b] M[b,c] ; 'L': dst[r,c] += a * sum_j M[r,j] src[j,c]
    #                                'LT': dst[r,c] += a * sum_k M[r,k] src[c,k] ; 'RT': dst[r,c] += a * sum_j src[j,r] M[j,c]  (source transposed)
    dst: Tuple[int, int, int, int, int]   # ch, r0, nr, c0, nc
    src: Tuple[int, int, int]             # ch, r0, c0
    mat: np.ndarray
    alpha: float = 1.0


@dataclass
class Rank1:
    dst_ch: int
    u: np.ndarray                  # [no_int, nv_int]
    src_ch: int
    v: np.ndarray                  # sigma_dst += u * <v, z_src>


@dataclass
class DiagTerm:
    ch: int
    d: np.ndarray                  # sigma += d o z


@dataclass
class SparseMap:
    """CSR rows -> (column, value): out[row] = sum_k val[k] * inp[col[k]]."""
    indptr: np.ndarray
    cols: np.ndarray
    vals: np.ndarray
    nrows: int


@dataclass
class Plan:
    method: str
    channels: List[ChannelSpec]
    k_terms: List[KTerm] = field(default_factory=list)
    kt_terms: List[KTermT] = field(default_factory=list)
    xc_scale: float = 1.0          # factor on the grid term (Z-vector plans: symmetrised densities)
    j_blocks: List[JBlock] = field(default_factory=list)
    j_mix: Optional[np.ndarray] = None
    xc_kind: str = "none"          # none | uks | alda0 | mcol | uks_tau | mcol_tau (meta-GGA tables with a tau component)
    local_gemms: List[LocalGemm] = field(default_factory=list)
    rank1s: List[Rank1] = field(default_factory=list)
    diags: List[DiagTerm] = field(default_factory=list)
    ext_dim: int = 0
    # entries (ext index, channel, i_int, a_int, coefficient): z_int[ch][i,a] = sum coef * z_ext[e]  and its transpose
    layout_entries: Optional[np.ndarray] = None     # structured: e, ch, i, a ; coef separately
    layout_coefs: Optional[np.ndarray] = None
    hdiag: Optional[np.ndarray] = None
    hdiag_needs_jdiag: Optional[dict] = None        # XSF: finish hdiag with J-block diagonals from the engine
    meta: dict = field(default_factory=dict)
    # keep what xtd_block_response reads (Coulomb Loo / Lvv of every channel, fp64 virtual MO values on the grid) resident
    block_response: bool = False

    def gather_map(self, ch: int) -> SparseMap:
        """ext -> internal block of channel `ch`, rows = i*nv_int + a."""
        c = self.channels[ch]
        ent, coef = self.layout_entries, self.layout_coefs
        sel = ent[:, 1] == ch
        rows = ent[sel, 2] * c.nv + ent[sel, 3]
        return _csr(rows, ent[sel, 0], coef[sel], c.no * c.nv)

    def scatter_map(self, offsets, lds) -> SparseMap:
        """internal (flat padded offsets) -> ext; offsets[ch], lds[ch] give the engine's block addresses."""
        ent, coef = self.layout_entries, self.layout_coefs
        off = np.asarray([offsets[c] for c in ent[:, 1]], dtype=np.int64)
        ld = np.asarray([lds[c] for c in ent[:, 1]], dtype=np.int64)
        cols = off + ent[:, 2] * ld + ent[:, 3]
        return _csr(ent[:, 0], cols, coef, self.ext_dim)


def _csr(rows, cols, vals, nrows) -> SparseMap:
    rows = np.asarray(rows, dtype=np.int64)
    order = np.argsort(rows, kind="stable")
    rows, cols, vals = rows[order], np.asarray(cols, dtype=np.int64)[order], np.asarray(vals, dtype=np.float64)[order]
    indptr = np.zeros(nrows + 1, dtype=np.int64)
    np.add.at(indptr, rows + 1, 1)
    return SparseMap(np.cumsum(indptr), cols, vals, nrows)


# --------------------------------------------------------------------------------------------------
# helpers
# --------------------------------------------------------------------------------------------------
def _two_block(n1: int, n2: int, first_mo: int):
    """internal positions [block1 (n1) | pad to even | block2 (n2)] -> (idx, blocks)"""
    off2 = _even(n1) if n2 > 0 else n1
    idx = np.full(off2 + n2, -1, dtype=np.int32)
    idx[:n1] = first_mo + np.arange(n1)
    idx[off2:off2 + n2] = first_mo + n1 + np.arange(n2)
    blocks = [(0, n1)] + ([(off2, n2)] if n2 > 0 else [])
    return idx, blocks


def _embed(mat, ridx_pos, cidx_pos, nr, ncol):
    """Place a matrix given on true indices into the padded internal index space."""
    out = np.zeros((nr, ncol))
    out[np.ix_(ridx_pos, cidx_pos)] = mat
    return out


def _pos(blocks):
    return np.concatenate([s + np.arange(n) for (s, n) in blocks]).astype(np.int64)


def _k_weight_tables(p: ProblemData, ch: int, nob: int, nvb: int, w0: np.ndarray) -> List[KTerm]:
    """exchange of A: -hyb K (+ -(alpha-hyb) K_lr), plus Delta-A weights w0 (full-range tensor only)."""
    out = []
    if not p.has_df:
        return out
    w = np.zeros((nob, nvb, nob, nvb)) if w0 is None else w0.copy()
    if p.hybrid:
        w -= p.hyb
    if np.any(w != 0):
        out.append(KTerm(0, ch, w))
    if p.hybrid and p.omega != 0.0 and p.has_df_lr:
        out.append(KTerm(1, ch, np.full((nob, nvb, nob, nvb), -(p.alpha - p.hyb))))
    return out


# --------------------------------------------------------------------------------------------------
# X-TDA
# --------------------------------------------------------------------------------------------------
def xtda_coeffs(s: float):
    r = math.sqrt((s + 1.0) / s)
    return 0.5 * (1 - r + 1 / (2 * s)), 0.5 * (-1 + r + 1 / (2 * s)), 0.5 / (2 * s)


def build_xtda_plan(p: ProblemData) -> Plan:
    nc, no, nv = p.nc, p.no, p.nv
    na, nb, nva, nvb = p.nocc_a, p.nocc_b, p.nvir_a, p.nvir_b
    # alpha: occ = [c | o] (two row blocks, rows need no padding but keep the even rule for transposed use), vir = v
    occ_a, ob_a = _two_block(nc, no, 0)
    vir_a = (na + np.arange(nva)).astype(np.int32)
    # beta: occ = c, vir = [o | pad | v]
    occ_b = np.arange(nb, dtype=np.int32)
    vir_b, vb_b = _two_block(no, nv, nb)
    cha = ChannelSpec(0, occ_a, 0, vir_a, ob_a, [(0, nva)])
    chb = ChannelSpec(1, occ_b, 1, vir_b, [(0, nb)], vb_b)
    plan = Plan("xtda", [cha, chb])
    oa_pos, va_pos = _pos(ob_a), np.arange(nva)
    ob_pos, vb_pos = np.arange(nb), _pos(vb_b)
    v2off = vb_b[1][0] if len(vb_b) > 1 else 0
    o2off = ob_a[1][0] if len(ob_a) > 1 else 0

    if p.has_df:
        for ci, chs in enumerate((cha, chb)):
            plan.k_terms += _k_weight_tables(p, ci, len(chs.o_blocks), len(chs.v_blocks), None)
        plan.j_blocks = [JBlock(0, 0, cha.no, 0, cha.nv), JBlock(1, 0, chb.no, 0, chb.nv)]
        plan.j_mix = np.ones((2, 2))
    plan.xc_kind = ("uks_tau" if p.xctype == "MGGA" else "uks") if p.xctype != "HF" else "none"

    fa, fb = p.fock_ks
    if p.restricted:
        # Fock blocks: sigma += z F_vv^T - F_oo z   (XTDA.py:629-632, 658-661)
        fvv_a = _embed(fa[na:, na:], va_pos, va_pos, cha.nv, cha.nv)
        foo_a = _embed(fa[:na, :na], oa_pos, oa_pos, cha.no, cha.no)
        fvv_b = _embed(fb[nb:, nb:], vb_pos, vb_pos, chb.nv, chb.nv)
        foo_b = _embed(fb[:nb, :nb], ob_pos, ob_pos, chb.no, chb.no)
        plan.local_gemms += [
            LocalGemm("R", (0, 0, cha.no, 0, cha.nv), (0, 0, 0), fvv_a.T.copy(), 1.0),
            LocalGemm("L", (0, 0, cha.no, 0, cha.nv), (0, 0, 0), foo_a, -1.0),
            LocalGemm("R", (1, 0, chb.no, 0, chb.nv), (1, 0, 0), fvv_b.T.copy(), 1.0),
            LocalGemm("L", (1, 0, chb.no, 0, chb.nv), (1, 0, 0), foo_b, -1.0),
        ]
        # spin-adaptation couplings between the CV blocks (XTDA.py:634-684)
        fha, fhb = p.fock_hf
        c1, c2, c3 = xtda_coeffs(p.spin_s)
        dvv = (fhb[na:, na:] - fha[na:, na:])           # nv x nv
        dcc = (fhb[:nb, :nb] - fha[:nb, :nb])           # nc x nc
        cva = (0, 0, nc, 0, nv)                          # CV(aa): rows c of alpha
        cvb = (1, 0, nc, v2off, nv)                      # CV(bb): cols v of beta
        plan.local_gemms += [
            LocalGemm("R", cva, (0, 0, 0), dvv.T.copy(), c1), LocalGemm("L", cva, (0, 0, 0), dcc, c2),
            LocalGemm("R", cva, (1, 0, v2off), dvv.T.copy(), -c3), LocalGemm("L", cva, (1, 0, v2off), dcc, -c3),
            LocalGemm("R", cvb, (1, 0, v2off), dvv.T.copy(), c2), LocalGemm("L", cvb, (1, 0, v2off), dcc, c1),
            LocalGemm("R", cvb, (0, 0, 0), dvv.T.copy(), -c3), LocalGemm("L", cvb, (0, 0, 0), dcc, -c3),
        ]
        da, db = fa.diagonal(), fb.diagonal()
    else:
        ea, eb = p.mo_energy
        e_a = ea[na:] - ea[:na, None]
        e_b = eb[nb:] - eb[:nb, None]
        plan.diags += [DiagTerm(0, _embed(e_a, oa_pos, va_pos, cha.no, cha.nv)),
                       DiagTerm(1, _embed(e_b, ob_pos, vb_pos, chb.no, chb.nv))]
        da, db = ea, eb
    e_a = da[na:] - da[:na, None]
    e_b = db[nb:] - db[:nb, None]
    plan.hdiag = np.hstack([e_a.ravel(), e_b.ravel()])

    # layout: PySCF order [alpha (i,a) | beta (i,a)]
    ia, aa = np.meshgrid(oa_pos, va_pos, indexing="ij")
    ib, ab = np.meshgrid(ob_pos, vb_pos, indexing="ij")
    n_a, n_b = na * nva, nb * nvb
    ent = np.zeros((n_a + n_b, 4), dtype=np.int64)
    ent[:, 0] = np.arange(n_a + n_b)
    ent[:n_a, 1], ent[:n_a, 2], ent[:n_a, 3] = 0, ia.ravel(), aa.ravel()
    ent[n_a:, 1], ent[n_a:, 2], ent[n_a:, 3] = 1, ib.ravel(), ab.ravel()
    plan.ext_dim = n_a + n_b
    plan.layout_entries, plan.layout_coefs = ent, np.ones(n_a + n_b)
    plan.meta = dict(nc=nc, no=no, nv=nv, o2off=o2off, v2off=v2off)
    return plan


# --------------------------------------------------------------------------------------------------
# spin-flip family: SF-TDA up/down, XSF-TDA (block or PySCF order, with/without the removed OO vector)
# --------------------------------------------------------------------------------------------------
def get_vect(no: int) -> np.ndarray:
    """Orthonormal basis of the OO space minus the trace vector (XSF_TDA.py:397-414): [no*no, no*no-1]."""
    vect = np.zeros((no, max(no - 1, 0)))
    for i in range(1, no):
        fac = 1.0 / math.sqrt((no - i + 1) * (no - i))
        vect[i - 1:, i - 1] = np.array([no - i] + [-1] * (no - i)) * fac
    vects = np.eye(no * no)[:, :-1].copy()
    for i in range(no - 1):
        vects[0::no + 1, i * (no + 1)] = vect[:, i]
    return vects


def xsf_factors(s: float):
    return (math.sqrt((2 * s + 1) / (2 * s)) - 1, math.sqrt((2 * s + 1) / (2 * s - 1)),
            math.sqrt((2 * s) / (2 * s - 1)) - 1, 1 / math.sqrt(2 * s * (2 * s - 1)))


def xsf_default_fglobal(p: ProblemData, method: int = 0, d_lda: float = 0.3, fit: bool = True) -> float:
    """XSF_TDA.py:1511-1518."""
    cx = p.hyb if p.omega == 0 else p.hyb + (p.alpha - p.hyb) * math.erf(p.omega)
    f = (1 - d_lda) * cx + d_lda
    if method == 1 and fit:
        f = f * 4 * (cx - 0.5) ** 2
    return f


def build_sf_plan(p: ProblemData, isf: int = -1, method: int = 0, sa: int = 0, layout: str = LAYOUT_PYSCF,
                  remove: bool = False, foo: float = 1.0, fglobal: Optional[float] = None,
                  hdiag_kind: str = "sf") -> Plan:
    """Spin-flip plans.

    isf=+1: SF-TDA up (beta occ -> alpha vir).  isf=-1: spin-flip down; sa>0 adds the XSF-TDA Delta A.
    hdiag_kind: 'sf' orbital-energy gaps (SF_TDA.py:208-217), 'xsf' Fock gaps + Delta-A diagonals in block
    order (XSF_TDA.py:915-961), 'gpu' Fock/orbital gaps in PySCF order (XSF_TDA_GPU.py:385-439).
    """
    nc, no, nv = p.nc, p.no, p.nv
    na, nb = p.nocc_a, p.nocc_b
    fa, fb = p.fock_ks
    xc_kind = {0: "alda0", 1: "mcol", 2: "none"}[method] if p.xctype != "HF" else "none"
    if xc_kind == "mcol" and p.xctype == "MGGA":
        xc_kind = "mcol_tau"           # the ALDA0 kernel has no tau part (SF_TDA.py:110-116: only rho_0 enters)
    if isf == 1:
        occ = np.arange(nb, dtype=np.int32)
        vir = (na + np.arange(nv)).astype(np.int32)
        ch = ChannelSpec(1, occ, 0, vir, [(0, nb)], [(0, nv)])
        plan = Plan("sf_up", [ch], xc_kind=xc_kind)
        plan.k_terms = _k_weight_tables(p, 0, 1, 1, None)
        plan.local_gemms = [LocalGemm("R", (0, 0, nb, 0, nv), (0, 0, 0), fa[na:, na:].T.copy(), 1.0),
                            LocalGemm("L", (0, 0, nb, 0, nv), (0, 0, 0), fb[:nb, :nb].copy(), -1.0)]
        if hdiag_kind == "gpu" and p.restricted:
            plan.hdiag = (fa.diagonal()[na:] - fb.diagonal()[:nb, None]).ravel()
        else:
            ea, eb = p.mo_energy
            plan.hdiag = (ea[na:] - eb[:nb, None]).ravel()
        ii, aa = np.meshgrid(np.arange(nb), np.arange(nv), indexing="ij")
        ent = np.stack([np.arange(nb * nv), np.zeros(nb * nv, dtype=np.int64), ii.ravel(), aa.ravel()], axis=1)
        plan.ext_dim, plan.layout_entries, plan.layout_coefs = nb * nv, ent.astype(np.int64), np.ones(nb * nv)
        plan.meta = dict(nc=nc, no=no, nv=nv)
        return plan

    # ---- spin-flip down: occ = alpha [c | pad | o], vir = beta [o | pad | v] --------------------------------
    occ_idx, o_blocks = _two_block(nc, no, 0)
    vir_idx, v_blocks = _two_block(no, nv, nb)
    ch = ChannelSpec(0, occ_idx, 1, vir_idx, o_blocks, v_blocks)
    o_pos, v_pos = _pos(o_blocks), _pos(v_blocks)
    o2off = o_blocks[1][0] if len(o_blocks) > 1 else 0
    v2off = v_blocks[1][0] if len(v_blocks) > 1 else 0
    nob, nvb = len(o_blocks), len(v_blocks)
    restricted_sa = sa if p.restricted else 0
    plan = Plan("xsf" if restricted_sa > 0 else "sf_down", [ch], xc_kind=xc_kind)
    if restricted_sa > 0:
        assert no >= 2, "XSF-TDA needs at least two open shells (2S-1 > 0)"
        assert nob == 2 and nvb == 2
    if fglobal is None:
        fglobal = xsf_default_fglobal(p, method)
    s = no / 2.0

    # Fock part of A (SF_TDA.py:234-240; XSF_TDA.py:1146-1169): sigma += z FB_vir^T - FA_occ z
    r_c = _embed(fb[nb:, nb:], v_pos, v_pos, ch.nv, ch.nv).T.copy()
    r_o = r_c.copy()
    l_o = -_embed(fa[:na, :na], o_pos, o_pos, ch.no, ch.no)
    l_v = l_o.copy()
    w_k = None
    if restricted_sa > 0:
        fha, fhb = p.fock_hf
        fs = (fhb - fha) * 0.5
        f1, f2, f3, f4 = xsf_factors(s)
        C, O, V = slice(0, nc), slice(nc, nc + no), slice(nc + no, None)
        # internal positions: occ c = [0,nc), occ o = o2off + [0,no); vir o = [0,no), vir v = v2off + [0,nv)
        oc, oo_ = np.arange(nc), o2off + np.arange(no)
        vo, vv = np.arange(no), v2off + np.arange(nv)
        fg = fglobal

        def add(mat, rows, cols, val):
            mat[np.ix_(rows, cols)] += val
        # SA >= 1 (XSF_TDA.py:1203-1212)
        add(r_c, vv, vv, fg * fs[V, V].T / s)                 # dcv += cv fs_vv / S
        add(l_v, oc, oc, fg * fs[C, C].T / s)                 # dcv += fs_cc^T cv / S   ("ji,xja->xia")
        add(l_o, oc, oc, fg * 2.0 * fs[C, C].T / (2 * s - 1))  # dco
        add(r_o, vv, vv, fg * 2.0 * fs[V, V].T / (2 * s - 1))  # dov  ("ab,xub->xua")
        w_k = np.zeros((2, 2, 2, 2))
        jm = np.zeros((2, 2))
        jm[0, 0] = jm[1, 1] = -fg / (2 * s - 1)               # -co_co^J, -ov_ov^J
        CVb, COb, OVb, OOb = (0, 1), (0, 0), (1, 1), (1, 0)   # (occ block, vir block)

        def kw(t, b, val):
            w_k[t[0], t[1], b[0], b[1]] += val
        if restricted_sa > 1:
            fhb_vo, fha_oc = fhb[V, O], fha[O, C]
            kw(CVb, COb, -fg * f1); kw(COb, CVb, -fg * f1); kw(CVb, OVb, -fg * f1); kw(OVb, CVb, -fg * f1)
            kw(COb, OVb, -fg / (2 * s - 1)); kw(OVb, COb, -fg / (2 * s - 1))
            jm[0, 1] = jm[1, 0] = fg / (2 * s - 1)
            add(r_c, vo, vv, fg * f1 * fhb_vo.T)              # dcv += f1 co F~b_vo^T   ("av,xiv->xia")
            add(r_c, vv, vo, fg * f1 * fhb_vo)                # dco += f1 cv F~b_vo     ("av,xja->xjv")
            add(l_v, oc, oo_, -fg * f1 * fha_oc.T)            # dcv -= f1 F~a_oc^T ov   ("vi,xva->xia")
            add(l_v, oo_, oc, -fg * f1 * fha_oc)              # dov -= f1 F~a_oc cv     ("vi,xib->xvb")
        if restricted_sa > 2:
            fha_co, fhb_co, fha_vo = fha[C, O], fhb[C, O], fha[V, O]
            kw(CVb, OOb, -fg * foo * (f2 - 1)); kw(OOb, CVb, -fg * foo * (f2 - 1))
            kw(COb, OOb, -fg * foo * f3); kw(OOb, COb, -fg * foo * f3)
            kw(OVb, OOb, -fg * foo * f3); kw(OOb, OVb, -fg * foo * f3)
            add(l_o, oc, oo_, -fg * foo * f3 * fha_co)        # dco -= f3 F~a_co oo     ("iw,xwu->xiu")
            add(l_o, oo_, oc, -fg * foo * f3 * fha_co.T)      # doo -= f3 F~a_co^T co   ("iw,xiv->xwv")
            add(r_o, vo, vv, fg * foo * f3 * fhb_vo.T)        # dov += f3 oo F~b_vo^T   ("av,xuv->xua")
            add(r_o, vv, vo, fg * foo * f3 * fhb_vo)          # doo += f3 ov F~b_vo     ("av,xwa->xwv")
            # trace terms: sigma += W <E,z> + E <W,z>,  E = identity on the OO block
            w = np.zeros((ch.no, ch.nv))
            w[np.ix_(oc, vv)] = fg * foo * (f2 / s) * fs[C, V]
            w[np.ix_(oc, vo)] = fg * foo * f4 * fhb_co
            w[np.ix_(oo_, vv)] = -fg * foo * f4 * fha_vo.T
            e = np.zeros((ch.no, ch.nv))
            e[oo_, vo] = 1.0
            plan.rank1s = [Rank1(0, w, 0, e), Rank1(0, e, 0, w)]
        if p.has_df:
            plan.j_blocks = [JBlock(0, 0, nc, 0, no), JBlock(0, o2off, no, v2off, nv)]     # co, ov
            plan.j_mix = jm
    plan.k_terms = _k_weight_tables(p, 0, nob, nvb, w_k)
    if restricted_sa == 0:
        # no block dependence: one full-range right and left product
        plan.local_gemms = [LocalGemm("R", (0, 0, ch.no, 0, ch.nv), (0, 0, 0), r_c, 1.0),
                            LocalGemm("L", (0, 0, ch.no, 0, ch.nv), (0, 0, 0), l_o, 1.0)]
    else:
        plan.local_gemms = [
            LocalGemm("R", (0, 0, nc, 0, ch.nv), (0, 0, 0), r_c, 1.0),
            LocalGemm("R", (0, o2off, no, 0, ch.nv), (0, o2off, 0), r_o, 1.0),
            LocalGemm("L", (0, 0, ch.no, 0, no), (0, 0, 0), l_o, 1.0),
            LocalGemm("L", (0, 0, ch.no, v2off, nv), (0, 0, v2off), l_v, 1.0),
        ]

    # ---- layouts ------------------------------------------------------------------------------------
    # true (i, a) with i in (c,o), a in (o,v)  ->  internal positions
    ii, aa = np.meshgrid(o_pos, v_pos, indexing="ij")             # [na, nvb]
    full_ext = np.arange(na * (no + nv)).reshape(na, no + nv)       # PySCF order index
    if layout == LAYOUT_BLOCK:
        blk = np.empty_like(full_ext)
        d1, d2, d3 = nc * nv, nc * nv + nc * no, nc * nv + nc * no + no * nv
        blk[:nc, no:] = np.arange(d1).reshape(nc, nv)
        blk[:nc, :no] = d1 + np.arange(nc * no).reshape(nc, no)
        blk[nc:, no:] = d2 + np.arange(no * nv).reshape(no, nv)
        blk[nc:, :no] = d3 + np.arange(no * no).reshape(no, no)
        full_ext = blk
    is_oo = np.zeros_like(full_ext, dtype=bool)
    is_oo[nc:, :no] = True
    if not remove:
        n = full_ext.size
        ent = np.stack([full_ext.ravel(), np.zeros(n, dtype=np.int64), ii.ravel(), aa.ravel()], axis=1)
        coef = np.ones(n)
        ext_dim = n
    else:
        assert no >= 2
        vects = get_vect(no)
        oo_ext_full = full_ext[nc:, :no].ravel()                  # ext index of OO element k (before removal)
        last = oo_ext_full[-1]
        # the shortened vector drops the LAST OO element of the layout; reduced coordinate m lives where OO element m was
        assert last == oo_ext_full.max()
        shift = lambda e: e - (e > last)
        rest = ~is_oo
        ent_rest = np.stack([shift(full_ext[rest]), np.zeros(rest.sum(), dtype=np.int64), ii[rest], aa[rest]], axis=1)
        kk, mm = np.nonzero(vects)                                # oo_full[k] = sum_m vects[k,m] oo_red[m]
        oo_i, oo_a = ii[nc:, :no].ravel(), aa[nc:, :no].ravel()
        ent_oo = np.stack([shift(oo_ext_full[mm]), np.zeros(kk.size, dtype=np.int64), oo_i[kk], oo_a[kk]], axis=1)
        ent = np.concatenate([ent_rest, ent_oo])
        coef = np.concatenate([np.ones(ent_rest.shape[0]), vects[kk, mm]])
        ext_dim = full_ext.size - 1
        plan.meta["vects"] = vects
    plan.ext_dim, plan.layout_entries, plan.layout_coefs = ext_dim, ent.astype(np.int64), coef

    # ---- preconditioner diagonal ----------------------------------------------------------------------
    if hdiag_kind == "sf":
        ea, eb = p.mo_energy
        h = (eb[nb:, None] - ea[:na]).T
        plan.hdiag = h.ravel()
    elif hdiag_kind == "gpu":
        da, db = (fa.diagonal(), fb.diagonal()) if p.restricted else (p.mo_energy[0], p.mo_energy[1])
        h = db[nb:] - da[:na, None]
        if remove:
            vects = plan.meta["vects"]
            hfull = h.ravel().copy()
            idx = np.arange(h.size).reshape(h.shape)
            oo_pos = idx[nc:, :no].ravel()
            hfull[oo_pos[:-1]] = h[nc:, :no].ravel() @ vects       # XSF_TDA_GPU.py:426-439
            plan.hdiag = np.delete(hfull, oo_pos[-1])
        else:
            plan.hdiag = h.ravel()
    elif hdiag_kind == "xsf":
        h = (fb.diagonal()[nb:][None, :] - fa.diagonal()[:na, None]).copy()
        pending = None
        if restricted_sa > 0:
            ds = ((p.fock_hf[1] - p.fock_hf[0]) * 0.5).diagonal()
            h[:nc, no:] += fglobal * (ds[nc + no:] + ds[:nc, None]) / s
            h[:nc, :no] += fglobal * (2.0 * ds[:nc, None]) / (2 * s - 1)
            h[nc:, no:] += fglobal * (2.0 * ds[nc + no:]) / (2 * s - 1)
            pending = dict(scale=-fglobal / (2 * s - 1))          # minus (iu|iu), (ua|ua) from the engine's J blocks
        plan.hdiag = h
        plan.hdiag_needs_jdiag = dict(pending=pending, remove=remove, nc=nc, no=no, nv=nv)
    else:
        raise ValueError(hdiag_kind)
    plan.meta.update(nc=nc, no=no, nv=nv, o2off=o2off, v2off=v2off, sa=restricted_sa, fglobal=fglobal, foo=foo,
                     layout=layout, remove=remove)
    return plan


def finish_xsf_hdiag(plan: Plan, co_j: Optional[np.ndarray], ov_j: Optional[np.ndarray]) -> np.ndarray:
    """Complete the XSF preconditioner (XSF_TDA.py:948-961, 999-1009) once the Coulomb diagonals
    (iu|iu) = sum_P L_iu^2 and (ua|ua) are known; returns block order (compressed if the OO vector is removed)."""
    info = plan.hdiag_needs_jdiag
    nc, no, nv = info["nc"], info["no"], info["nv"]
    h = plan.hdiag.copy()
    if info["pending"] is not None:
        h[:nc, :no] += info["pending"]["scale"] * co_j
        h[nc:, no:] += info["pending"]["scale"] * ov_j
    hd = np.hstack([h[:nc, no:].ravel(), h[:nc, :no].ravel(), h[nc:, no:].ravel(), h[nc:, :no].ravel()])
    if info["remove"]:
        vects = plan.meta["vects"]
        d3 = nc * nv + nc * no + no * nv
        hd = np.hstack([hd[:d3], np.einsum("x,xy,xy->y", hd[d3:], vects, vects)])
    return hd


# --------------------------------------------------------------------------------------------------
# Z-vector (coupled-perturbed) operator of the spin-flip-up TDA gradients  (SURVEY 8f row f3)
# --------------------------------------------------------------------------------------------------
def zvector_sym_fock(p: ProblemData) -> dict:
    """Symmetrised MO Fock blocks of the ROKS orbital Hessian (grad_hb/tdroks_sfu.py:224-234)."""
    nc, no = p.nc, p.no
    fa, fb = p.fock_ks
    C, O, V = slice(0, nc), slice(nc, nc + no), slice(nc + no, None)
    sym = lambda f, r, c: 0.5 * (f[r, c] + f[c, r].T)
    return dict(acc=sym(fa, C, C), aoc=sym(fa, O, C), avc=sym(fa, V, C), avv=sym(fa, V, V), aoo=sym(fa, O, O),
                bcc=sym(fb, C, C), bvc=sym(fb, V, C), bvv=sym(fb, V, V), bvo=sym(fb, V, O), boo=sym(fb, O, O))


def build_zvector_plan(p: ProblemData, with_diag: bool = True) -> Plan:
    """The linear operator of the Z-vector equation as an engine plan.

    ROKS reference (`p.restricted`): `matvec` of grad_hb/tdroks_sfu.py:284-321 -- the ROHF orbital Hessian on the rotations
    x = [vc (nv x nc) | vo (nv x no) | oc (no x nc)] (virtual-major blocks):  F-couplings - 2 G[Z^S], where G is the hermi = 1
    response `vresp` (tdroks_sfu.py:283,295) of the symmetrised density (dm + dm^T)/2 projected on the occupied-virtual blocks.
    UKS reference: `fvind` of grad_hb/tduks_sfu.py:249-258 on x = [alpha (nv x nocc_a) | beta (nvir_b x nocc_b)], G[dm + dm^T];
    `with_diag` adds the orbital-energy differences, i.e. the operator `ucphf.solve` inverts (tduks_sfu.py:261-263).

    In the engine's MO-resident vocabulary the response of a symmetrised trial density is the TDA response (direct exchange,
    Coulomb, grid kernel -- the X-TDA plan's terms) plus the exchange of the TRANSPOSED density (`KTermT`):
        K[dm + dm^T]_ai = sum_P sum_jb (L_ab L_ij + L_aj L_ib) z_jb ,   J and f_xc just double.
    """
    nc, no, nv = p.nc, p.no, p.nv
    na, nb, nva, nvb = p.nocc_a, p.nocc_b, p.nvir_a, p.nvir_b
    occ_a, ob_a = _two_block(nc, no, 0)
    vir_a = (na + np.arange(nva)).astype(np.int32)
    occ_b = np.arange(nb, dtype=np.int32)
    vir_b, vb_b = _two_block(no, nv, nb)
    cha = ChannelSpec(0, occ_a, 0, vir_a, ob_a, [(0, nva)])
    chb = ChannelSpec(1, occ_b, 1, vir_b, [(0, nb)], vb_b)
    plan = Plan("zvector_roks" if p.restricted else "zvector_uks", [cha, chb])
    oa_pos, va_pos = _pos(ob_a), np.arange(nva)
    ob_pos, vb_pos = np.arange(nb), _pos(vb_b)
    v2off = vb_b[1][0] if len(vb_b) > 1 else 0
    o2off = ob_a[1][0] if len(ob_a) > 1 else 0
    # G[dm + dm^T] = g * (2 J + 2 f_xc - hyb (K + K^T-type));  ROKS: -2 G[(dm + dm^T)/2]  ->  g = -1;  UKS: g = +1
    g = -1.0 if p.restricted else 1.0
    if p.has_df:
        plan.j_blocks = [JBlock(0, 0, cha.no, 0, cha.nv), JBlock(1, 0, chb.no, 0, chb.nv)]
        plan.j_mix = 2.0 * g * np.ones((2, 2))
        if p.hybrid:
            for ci, chs in enumerate((cha, chb)):
                shape = (len(chs.o_blocks), len(chs.v_blocks)) * 2
                plan.k_terms.append(KTerm(0, ci, np.full(shape, -g * p.hyb)))
                plan.kt_terms.append(KTermT(0, ci, -g * p.hyb))
                if p.omega != 0.0 and p.has_df_lr:
                    plan.k_terms.append(KTerm(1, ci, np.full(shape, -g * (p.alpha - p.hyb))))
                    plan.kt_terms.append(KTermT(1, ci, -g * (p.alpha - p.hyb)))
    if p.xctype != "HF":
        plan.xc_kind = "uks_tau" if p.xctype == "MGGA" else "uks"
        plan.xc_scale = 2.0 * g

    if p.restricted:
        f = zvector_sym_fock(p)
        cva, ova = (0, 0, nc, 0, nv), (0, o2off, no, 0, nv)         # alpha: rows c / rows o
        cvb, cob = (1, 0, nc, v2off, nv), (1, 0, nc, 0, no)         # beta: cols v / cols o
        lg = plan.local_gemms
        # Fxvc (tdroks_sfu.py:301-308), split over the two channels that carry the vc block
        lg += [LocalGemm("R", cva, (0, 0, 0), f["avv"].T.copy(), -1.0), LocalGemm("L", cva, (0, 0, 0), f["acc"].T.copy(), 1.0),
               LocalGemm("L", cva, (0, o2off, 0), f["aoc"].T.copy(), 1.0),
               LocalGemm("R", cvb, (1, 0, v2off), f["bvv"].T.copy(), -1.0), LocalGemm("L", cvb, (1, 0, v2off), f["bcc"].T.copy(), 1.0),
               LocalGemm("R", cvb, (1, 0, 0), f["bvo"].T.copy(), -1.0)]
        if no > 0:
            # Fxvo (:309-314): the oc block of the beta channel enters transposed
            lg += [LocalGemm("RT", ova, (1, 0, 0), f["bvc"].T.copy(), -1.0), LocalGemm("L", ova, (0, 0, 0), f["aoc"].copy(), 1.0),
                   LocalGemm("R", ova, (0, o2off, 0), f["avv"].copy(), -1.0), LocalGemm("L", ova, (0, o2off, 0), f["aoo"].copy(), 1.0)]
            # Fxoc (:315-320): the vo block of the alpha channel enters transposed
            lg += [LocalGemm("R", cob, (1, 0, 0), f["boo"].T.copy(), -1.0), LocalGemm("L", cob, (1, 0, 0), f["bcc"].copy(), 1.0),
                   LocalGemm("R", cob, (1, 0, v2off), f["bvo"].copy(), -1.0), LocalGemm("LT", cob, (0, o2off, 0), f["avc"].T.copy(), 1.0)]
        d = lambda m: np.diagonal(m)
        h_vc = -(d(f["avv"]) + d(f["bvv"]))[:, None] + (d(f["acc"]) + d(f["bcc"]))[None, :]
        h_vo = -d(f["avv"])[:, None] + d(f["aoo"])[None, :]
        h_oc = -d(f["boo"])[:, None] + d(f["bcc"])[None, :]
        plan.hdiag = np.hstack([h_vc.ravel(), h_vo.ravel(), h_oc.ravel()])
        # layout: x = [vc (a,i) | vo (a,t) | oc (t,i)]; the vc block feeds both channels and collects from both
        a_, i_ = np.meshgrid(np.arange(nv), np.arange(nc), indexing="ij")
        e_vc = (a_ * nc + i_).ravel()
        ent = [np.stack([e_vc, np.zeros_like(e_vc), oa_pos[i_.ravel()], va_pos[a_.ravel()]], axis=1),
               np.stack([e_vc, np.ones_like(e_vc), ob_pos[i_.ravel()], vb_pos[no + a_.ravel()]], axis=1)]
        if no > 0:
            a_, t_ = np.meshgrid(np.arange(nv), np.arange(no), indexing="ij")
            e_vo = (nv * nc + a_ * no + t_).ravel()
            ent.append(np.stack([e_vo, np.zeros_like(e_vo), oa_pos[nc + t_.ravel()], va_pos[a_.ravel()]], axis=1))
            t_, i_ = np.meshgrid(np.arange(no), np.arange(nc), indexing="ij")
            e_oc = (nv * nc + nv * no + t_ * nc + i_).ravel()
            ent.append(np.stack([e_oc, np.ones_like(e_oc), ob_pos[i_.ravel()], vb_pos[t_.ravel()]], axis=1))
        ent = np.concatenate(ent).astype(np.int64)
        plan.ext_dim = nv * nc + nv * no + no * nc
    else:
        ea, eb = p.mo_energy
        e_a = ea[na:, None] - ea[None, :na]                       # [nv, nocc_a]  virtual-major like the vectors
        e_b = eb[nb:, None] - eb[None, :nb]
        plan.hdiag = np.hstack([e_a.ravel(), e_b.ravel()])
        if with_diag:
            plan.diags += [DiagTerm(0, _embed(e_a.T, oa_pos, va_pos, cha.no, cha.nv)),
                           DiagTerm(1, _embed(e_b.T, ob_pos, vb_pos, chb.no, chb.nv))]
        a_, i_ = np.meshgrid(np.arange(nva), np.arange(na), indexing="ij")
        e1 = (a_ * na + i_).ravel()
        a2, i2 = np.meshgrid(np.arange(nvb), np.arange(nb), indexing="ij")
        e2 = (nva * na + a2 * nb + i2).ravel()
        ent = np.concatenate([np.stack([e1, np.zeros_like(e1), oa_pos[i_.ravel()], va_pos[a_.ravel()]], axis=1),
                              np.stack([e2, np.ones_like(e2), ob_pos[i2.ravel()], vb_pos[a2.ravel()]], axis=1)]).astype(np.int64)
        plan.ext_dim = nva * na + nvb * nb
    plan.layout_entries, plan.layout_coefs = ent, np.ones(ent.shape[0])
    plan.meta = dict(nc=nc, no=no, nv=nv, o2off=o2off, v2off=v2off)
    return plan


# --------------------------------------------------------------------------------------------------
# Right-hand side of the Z-vector equation: responses of densities with occupied-occupied / virtual-virtual blocks
# --------------------------------------------------------------------------------------------------
def build_mo_response_plan(p: ProblemData, range_separated: bool = True) -> Plan:
    """`vresp(D)` for ARBITRARY MO-basis densities, all blocks out: one "vector" is [T_a (nmo x nmo) | T_b (nmo x nmo)] row-major,
    D_s = C_s T_s C_s^T, and the result is C_s^T (f_xc[D] + J[D_a + D_b] - hyb K[D_s]) C_s in the same layout.

    The channels of the engine are index SETS, not "occupied" and "virtual": with both sets = all MOs of a spin the direct exchange
    term is the general K build, a full-width Coulomb block the general J build and the MO-on-grid contraction the general f_xc
    response.  This is what the Q matrix of the gradients needs for the relaxed difference densities T (virtual-virtual block for
    alpha, occupied-occupied for beta: `mf.get_jk(mol, (dmzvva, dmzoob), hermi=1)` + `f1oo`, grad_hb/tdroks_sfu.py:241-251,
    tduks_sfu.py:219-229) and the W matrix for the occupied-occupied projection of G[Z^S] (:339-351).  A one-off per state, so the
    MO-resident tensor of the whole MO space (naux x nmo^2 per spin) is affordable up to ~1000 basis functions on one GPU; shard beyond.
    `range_separated=False` leaves the long-range exchange out, as the reference's Q matrix does (`vk * hyb` only, tdroks_sfu.py:247-251)."""
    nmo = p.nmo
    idx = np.arange(nmo, dtype=np.int32)
    chs = [ChannelSpec(s, idx.copy(), s, idx.copy(), [(0, nmo)], [(0, nmo)]) for s in (0, 1)]
    plan = Plan("mo_response", chs)
    if p.has_df:
        plan.j_blocks = [JBlock(0, 0, nmo, 0, nmo), JBlock(1, 0, nmo, 0, nmo)]
        plan.j_mix = np.ones((2, 2))
        if p.hybrid:
            for ci in (0, 1):
                plan.k_terms.append(KTerm(0, ci, np.full((1, 1, 1, 1), -p.hyb)))
                if range_separated and p.omega != 0.0 and p.has_df_lr:
                    plan.k_terms.append(KTerm(1, ci, np.full((1, 1, 1, 1), -(p.alpha - p.hyb))))
    if p.xctype != "HF":
        plan.xc_kind = "uks_tau" if p.xctype == "MGGA" else "uks"
    n2 = nmo * nmo
    ii, aa = np.meshgrid(np.arange(nmo), np.arange(nmo), indexing="ij")
    ent = np.concatenate([np.stack([s * n2 + np.arange(n2), np.full(n2, s), ii.ravel(), aa.ravel()], axis=1) for s in (0, 1)])
    plan.ext_dim, plan.layout_entries, plan.layout_coefs = 2 * n2, ent.astype(np.int64), np.ones(2 * n2)
    plan.hdiag = np.ones(2 * n2)
    plan.meta = dict(nmo=nmo)
    return plan


def build_mo_sf_exchange_plan(p: ProblemData) -> Plan:
    """K[X] of a spin-flip density X = C_b z C_a^T in the mixed MO basis: one "vector" is z (nmo_b x nmo_a) row-major, the result is
    C_b^T K[X] C_a (`mf.get_k(mol, dmt, hermi=0)` projected as `veff0mo`, grad_hb/tdroks_sfu.py:249-254; unscaled: multiply by hyb)."""
    nmo = p.nmo
    idx = np.arange(nmo, dtype=np.int32)
    plan = Plan("mo_sf_exchange", [ChannelSpec(1, idx.copy(), 0, idx.copy(), [(0, nmo)], [(0, nmo)])])
    plan.k_terms = [KTerm(0, 0, np.ones((1, 1, 1, 1)))]
    n2 = nmo * nmo
    ii, aa = np.meshgrid(np.arange(nmo), np.arange(nmo), indexing="ij")
    ent = np.stack([np.arange(n2), np.zeros(n2, dtype=np.int64), ii.ravel(), aa.ravel()], axis=1)
    plan.ext_dim, plan.layout_entries, plan.layout_coefs = n2, ent.astype(np.int64), np.ones(n2)
    plan.hdiag = np.ones(n2)
    plan.meta = dict(nmo=nmo)
    return plan
