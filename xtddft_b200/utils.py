"""Amplitude layouts and labels returned by the driver classes (host-side integer permutations and tiny fp64 maps).

Same contracts as the reference helpers: `order_pyscf2my`, `so2st`, `st2so` (xtddft/utils/utils.py:44-122),
`deal_v_davidson` (xtddft/SF_TDA.py:304-345, xtddft/XSF_TDA.py:1419-1453), the Delta<S^2> labels (xtddft/XTDA.py:831-836,
xtddft/SF_TDA.py:819-825).  SURVEY Appendix A.5.
"""
from __future__ import annotations

import numpy as np

from .plan import get_vect  # noqa: F401  (re-exported: XSF_TDA.get_vect)

ha2eV = 27.2113834          # xtddft/utils/unit.py:7 (X-TDA, SF-TDA, GPU classes)
au2ev_xsf = 27.21138505     # xtddft/XSF_TDA.py:21


def order_pyscf2my(nc: int, no: int, nv: int) -> np.ndarray:
    """PySCF order [alpha (c,o) x v | beta c x (o,v)] -> [CV(aa) | OV(aa) | CO(bb) | CV(bb)]."""
    na = (nc + no) * nv
    beta = na + np.arange(nc * (no + nv)).reshape(nc, no + nv)
    return np.concatenate([np.arange(na), beta[:, :no].ravel(), beta[:, no:].ravel()])


def _split_my(v, nc, no, nv):
    d1, d2, d3 = nc * nv, (nc + no) * nv, (nc + no) * nv + nc * no
    return v[:d1], v[d1:d2], v[d2:d3], v[d3:]


def cvs_rows(nc: int, no: int, nv: int, core_a, core_b) -> np.ndarray:
    """Rows of the core-valence-separated X-TDA layout inside the full PySCF order: [alpha (i in core_a, a) | beta (i in core_b, a)],
    the order of `plan.build_xtda_plan(p, core)`."""
    na, nvb = nc + no, no + nv
    ra = (np.asarray(core_a, dtype=np.int64)[:, None] * nv + np.arange(nv)).ravel()
    rb = na * nv + (np.asarray(core_b, dtype=np.int64)[:, None] * nvb + np.arange(nvb)).ravel()
    return np.concatenate([ra, rb])


def cvs_embed(x, rows, dim: int) -> np.ndarray:
    """Vectors on the rows `rows` of a `dim`-row layout (first axis) zero-padded to the whole layout."""
    x = np.asarray(x)
    out = np.zeros((dim,) + x.shape[1:], dtype=x.dtype)
    out[rows] = x
    return out


def cvs_order_pyscf2my(nc: int, no: int, nv: int, core_a, core_b):
    """(order, my_rows): `x[order]` takes core-valence-separated vectors from PySCF order to the order of `order_pyscf2my`
    restricted to the core rows [CV(aa) | OV(aa) | CO(bb) | CV(bb)]; `my_rows` are those rows inside the full order_pyscf2my layout."""
    rows = cvs_rows(nc, no, nv, core_a, core_b)
    full = order_pyscf2my(nc, no, nv)
    inv = np.full(full.size, -1, dtype=np.int64)
    inv[rows] = np.arange(rows.size)
    sel = inv[full]
    keep = sel >= 0
    return sel[keep], np.nonzero(keep)[0]


def so2st(eigvec, nc, no, nv, core=None):
    """Spin-orbital -> singlet / triplet combinations of the CV blocks.  `core = (core_a, core_b)`: `eigvec` holds core-valence-
    separated vectors in `cvs_order_pyscf2my` order; the result is the full-space so2st of the zero-padded vectors, on the core rows.
    The singlet / triplet pairs stay on the core rows only when the closed alpha core rows are exactly the beta core rows."""
    if core is not None:
        core_a, core_b = (np.asarray(c) for c in core)
        if not np.array_equal(core_a[core_a < nc], core_b):
            raise ValueError("so2st: the closed-shell alpha core orbitals must be the beta core orbitals")
        _, my_rows = cvs_order_pyscf2my(nc, no, nv, core_a, core_b)
        full = cvs_embed(eigvec, my_rows, (nc + no) * nv + nc * (no + nv))
        return so2st(full, nc, no, nv)[my_rows]
    cva, ova, cob, cvb = _split_my(eigvec, nc, no, nv)
    r = np.sqrt(2.0) / 2.0
    return np.concatenate((r * (cva + cvb), ova, cob, r * (cva - cvb)), axis=0)


def st2so(eigvec, nc, no, nv):
    cv0, ov0, co0, cv1 = _split_my(eigvec, nc, no, nv)
    return np.concatenate(((cv0 + cv1) / np.sqrt(2.0), ov0, co0, (cv0 - cv1) / np.sqrt(2.0)), axis=0)


def sf_pyscf_to_block(nc: int, no: int, nv: int) -> np.ndarray:
    """spin-flip-down PySCF order ((c,o) x (o,v), row-major) -> [cv | co | ov | oo]."""
    idx = np.arange((nc + no) * (no + nv)).reshape(nc + no, no + nv)
    return np.concatenate([idx[:nc, no:].ravel(), idx[:nc, :no].ravel(), idx[nc:, no:].ravel(), idx[nc:, :no].ravel()])


def deal_v_davidson(v, nc: int, no: int, nv: int, removed: bool = False):
    """Columns of `v` from PySCF order (optionally without the last OO element) to block order."""
    v = np.asarray(v)
    if not removed:
        return v[sf_pyscf_to_block(nc, no, nv)]
    full = np.arange((nc + no) * (no + nv)).reshape(nc + no, no + nv)
    last = full[nc + no - 1, no - 1]
    sh = lambda a: a - (a > last)
    parts = [full[:nc, no:].ravel(), full[:nc, :no].ravel(), full[nc:, no:].ravel(), full[nc:, :no].ravel()[:-1]]
    return v[np.concatenate([sh(p) for p in parts])]


def delta_s2_xtda(v_my, nc, no, nv):
    cva, _, _, cvb = _split_my(v_my, nc, no, nv)
    return np.einsum("ik,ik->k", cva - cvb, cva - cvb)


def delta_s2_sf_roks(v_block, nc, no, nv, vects=None):
    """ROKS reference, spin-flip down: dS2 = -no + 1 + |cv|^2 - |oo|^2 + (tr oo)^2."""
    d1, d3 = nc * nv, nc * nv + nc * no + no * nv
    out = np.empty(v_block.shape[1])
    for k in range(v_block.shape[1]):
        cv = v_block[:d1, k]
        oo = v_block[d3:, k]
        if vects is not None:
            oo = vects @ oo
        oo = oo.reshape(no, no)
        out[k] = -no + 1 + cv @ cv - np.sum(oo * oo) + np.trace(oo) ** 2
    return out
