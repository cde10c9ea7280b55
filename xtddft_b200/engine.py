"""SigmaEngine: the host-side owner of one libxtdsigma engine on one B200.

PyTorch is used only for buffer ownership (device tensors whose raw pointers cross the C-ABI), stream
identity and the NCCL process group.  All arithmetic of the sigma path runs in hand-written sm_100a kernels
inside libxtdsigma.so; if the library is missing, construction fails (no CPU fallback).

    eng = SigmaEngine.from_problem(plan, problem)      # upload once per solve
    hz  = eng.sigma(z)                                 # z: torch cuda [nvec, dim] -> torch cuda [nvec, dim]
    vind = eng.as_vind()                               # NumPy-in / NumPy-out callable with the reference's `vind` contract
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional

import numpy as np

from . import _lib
from .dist import SigmaReducer, split_range
from .plan import Plan, finish_xsf_hdiag
from .problem import ProblemData

_KIND = {"none": _lib.XTD_FXC_NONE, "uks": _lib.XTD_FXC_UKS, "alda0": _lib.XTD_FXC_ALDA0, "mcol": _lib.XTD_FXC_MCOL,
         "uks_tau": _lib.XTD_FXC_UKS_TAU, "mcol_tau": _lib.XTD_FXC_MCOL_TAU}      # *_tau: meta-GGA kernel tables (5 components)


def _ptr(t) -> C.c_void_p:
    return C.c_void_p(t.data_ptr())


def _np_ptr(a: np.ndarray) -> C.c_void_p:
    return C.c_void_p(a.ctypes.data)


def _pad16(n: int) -> int:
    return (max(n, 1) + 15) // 16 * 16


class SigmaEngine:
    def __init__(self, plan: Plan, nao: int, mo_coeff: np.ndarray, *, workspace_bytes: int = 2 << 30, device=None,
                 reducer: Optional[SigmaReducer] = None, exchange_slices: Optional[int] = None):
        import torch
        if not torch.cuda.is_available():
            raise _lib.XtdError("SigmaEngine needs a CUDA device (sm_100a); there is no CPU fallback")
        self.torch = torch
        self.lib = _lib.load()
        self.plan = plan
        self.nao = int(nao)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        torch.cuda.set_device(self.device)
        self.reducer = reducer
        self._keep: List[object] = []          # device tensors the engine holds raw pointers to
        self._grid_keep: List[object] = []     # ... only until grid_commit
        self._h = C.c_void_p()
        _lib.check(self.lib.xtd_create(C.byref(self._h), self.nao, int(workspace_bytes)), "xtd_create")
        self._set_stream()
        # exchange contraction of uniform-weight terms: 0 = FP64 DMMA, 3..8 = INT8 tensor-core emulation with that many
        # radix-256 digit planes (csrc/ozaki.cuh).  None: the XTD_OZAKI environment variable, else FP64 DMMA.
        if exchange_slices is None:
            env = os.environ.get("XTD_OZAKI", "")
            if env != "":
                exchange_slices = int(env)
            else:
                # default: 6 planes (46 bits below each row scale, ~4e-12 on sigma, 4x the DMMA rate) once the virtual block spans
                # several 128-column tiles; small problems are launch-bound and stay on the FP64 DMMA GEMM
                big = max((len(ch.vir_idx) for ch in plan.channels), default=0) >= 512
                exchange_slices = 6 if big else 0
        self.exchange_slices = int(exchange_slices)
        if self.exchange_slices:
            _lib.check(self.lib.xtd_set_exchange_emulation(self._h, self.exchange_slices), "xtd_set_exchange_emulation")
        if plan.block_response:
            _lib.check(self.lib.xtd_enable_block_response(self._h), "xtd_enable_block_response")
        self.finalized = False
        self.max_nvec = 0
        self.ext_dim = int(plan.ext_dim)
        self._naux_total = [0, 0]
        # orbitals
        mo_coeff = np.ascontiguousarray(mo_coeff, dtype=np.float64)
        for spin in (0, 1):
            c = torch.from_numpy(mo_coeff[spin]).to(self.device)
            self._keep.append(c)
            _lib.check(self.lib.xtd_set_mo(self._h, spin, _ptr(c), c.shape[1], c.shape[1]), "xtd_set_mo")
        # channels
        for ch in plan.channels:
            occ = np.ascontiguousarray(ch.occ_idx, dtype=np.int32)
            vir = np.ascontiguousarray(ch.vir_idx, dtype=np.int32)
            ob = np.ascontiguousarray(np.array(ch.o_blocks, dtype=np.int32).ravel())
            vb = np.ascontiguousarray(np.array(ch.v_blocks, dtype=np.int32).ravel())
            _lib.check(self.lib.xtd_add_channel(self._h, ch.spin_o, _np_ptr(occ), len(occ), ch.spin_v, _np_ptr(vir), len(vir),
                                                _np_ptr(ob), len(ch.o_blocks), _np_ptr(vb), len(ch.v_blocks)), "xtd_add_channel")
        # exchange terms and Coulomb blocks must be declared before the tensor is streamed in
        for kt in plan.k_terms:
            w = np.ascontiguousarray(kt.weights, dtype=np.float64)
            _lib.check(self.lib.xtd_add_kterm(self._h, kt.tensor, kt.ch, _np_ptr(w), w.shape[0], w.shape[1]), "xtd_add_kterm")
        for kt in plan.kt_terms:
            _lib.check(self.lib.xtd_add_kterm_t(self._h, kt.tensor, kt.ch, float(kt.weight)), "xtd_add_kterm_t")
        for jb in plan.j_blocks:
            _lib.check(self.lib.xtd_add_jblock(self._h, jb.ch, jb.r0, jb.nr, jb.c0, jb.nc), "xtd_add_jblock")
        if plan.j_blocks:
            m = np.ascontiguousarray(plan.j_mix, dtype=np.float64)
            _lib.check(self.lib.xtd_set_jmix(self._h, _np_ptr(m), m.shape[0]), "xtd_set_jmix")
        self.tensors_used = sorted({kt.tensor for kt in plan.k_terms} | {kt.tensor for kt in plan.kt_terms} | ({0} if plan.j_blocks else set()))

    # ---- plumbing ---------------------------------------------------------------------------------
    def _set_stream(self):
        s = self.torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(self.lib.xtd_set_stream(self._h, C.c_void_p(s)), "xtd_set_stream")

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self.lib.xtd_destroy(self._h)
            self._h = C.c_void_p()
        self._keep = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- density fitting ----------------------------------------------------------------------------
    def df_begin(self, tensor: int, naux_local: int):
        _lib.check(self.lib.xtd_df_begin(self._h, tensor, int(naux_local)), "xtd_df_begin")
        self._df_left = getattr(self, "_df_left", {})
        self._df_carry = getattr(self, "_df_carry", {})
        self._df_left[tensor] = int(naux_local)
        self._df_carry[tensor] = None

    def df_add(self, tensor: int, chunk, packed: bool = False):
        """chunk: torch cuda fp64 [np, nao, nao] (any row stride) or packed lower-triangular [np, nao(nao+1)/2]."""
        assert chunk.is_cuda and chunk.dtype == self.torch.float64
        if self.exchange_slices:
            # emulated exchange: the library wants whole scale groups (<= 4 aux functions) in every chunk but the last;
            # carry the remainder of a ragged chunk over to the next call
            carry = self._df_carry.get(tensor)
            if carry is not None:
                chunk = self.torch.cat([carry, chunk], dim=0)
                self._df_carry[tensor] = None
            n = chunk.shape[0]
            if n < self._df_left[tensor] and n % 12:
                keep = n // 12 * 12                      # a multiple of every group size (1, 2, 3, 4)
                self._df_carry[tensor] = chunk[keep:].clone()
                chunk = chunk[:keep]
                if keep == 0:
                    return
            self._df_left[tensor] -= chunk.shape[0]
        if packed:
            assert chunk.dim() == 2 and chunk.stride(1) == 1
            _lib.check(self.lib.xtd_df_add(self._h, tensor, _ptr(chunk), chunk.shape[0], 0, chunk.stride(0), 1), "xtd_df_add")
        else:
            assert chunk.dim() == 3 and chunk.stride(2) == 1
            _lib.check(self.lib.xtd_df_add(self._h, tensor, _ptr(chunk), chunk.shape[0], chunk.stride(1), chunk.stride(0), 0),
                       "xtd_df_add")

    # ---- ROHF-form Fock difference (setup stage, SURVEY 8f row f2) ------------------------------------------------------
    def set_open_orbitals(self, spin: int, open_idx):
        """Declare the open-shell MOs before the tensor streams in: the library then accumulates K[D_open] in the MO basis."""
        idx = np.ascontiguousarray(open_idx, dtype=np.int32)
        _lib.check(self.lib.xtd_set_open_orbitals(self._h, int(spin), _np_ptr(idx), len(idx)), "xtd_set_open_orbitals")
        self._kopen_nmo = int(self._keep[spin].shape[1])

    def kopen(self) -> np.ndarray:
        """K[D_open][p][q] = sum_P sum_u L^P_pu L^P_qu = F_beta^HF - F_alpha^HF of the ROHF-form Fock matrices (XTDA.py:607-613,
        XSF_TDA.py:1103-1111), all-reduced over the aux shards."""
        torch = self.torch
        n = self._kopen_nmo
        out = torch.zeros((n, n), dtype=torch.float64, device=self.device)
        self._set_stream()
        _lib.check(self.lib.xtd_get_kopen(self._h, _ptr(out), n), "xtd_get_kopen")
        if self.reducer is not None:
            self.reducer.allreduce_(out)
        return out.cpu().numpy()

    def load_cderi(self, tensor: int, cderi: np.ndarray, chunk: int = 64):
        """Stream a host tensor [naux_local, nao, nao] through the device in aux chunks."""
        torch = self.torch
        naux = cderi.shape[0]
        self.df_begin(tensor, naux)
        for p0 in range(0, naux, chunk):
            blk = torch.from_numpy(np.ascontiguousarray(cderi[p0:p0 + chunk])).to(self.device)
            self.df_add(tensor, blk)

    def load_cderi_packed(self, tensor: int, src, naux: int, rank: int = 0, world: int = 1, chunk: int = 64):
        """Stream lower-triangular packed rows [naux, nao(nao+1)/2] (PySCF `with_df._cderi`): `src` is a 2-D host array or a
        zero-argument callable returning an iterator of row blocks (`with_df.loop()`); this rank keeps rows [p0, p1)."""
        torch = self.torch
        p0, p1 = split_range(int(naux), rank, world)
        self.df_begin(tensor, p1 - p0)
        blocks = src() if callable(src) else (src[i:i + chunk] for i in range(0, src.shape[0], chunk))
        row = 0
        for blk in blocks:
            blk = np.asarray(blk)
            lo, hi = max(p0 - row, 0), min(p1 - row, blk.shape[0])
            row += blk.shape[0]
            for i in range(lo, hi, chunk):
                part = torch.from_numpy(np.ascontiguousarray(blk[i:min(i + chunk, hi)], dtype=np.float64)).to(self.device)
                self.df_add(tensor, part, packed=True)

    # ---- grid ---------------------------------------------------------------------------------------
    def set_grid(self, ao, weights):
        """ao: torch cuda [nvar, ng, nao(+pad)] fp64, weights: torch cuda [ng]."""
        torch = self.torch
        nvar, ng, n = ao.shape
        if ao.stride(2) != 1 or ao.stride(1) % 2 or ao.stride(0) % 2 or ao.data_ptr() % 16:
            ld = _pad16(self.nao)
            buf = torch.zeros((nvar, ng, ld), dtype=torch.float64, device=self.device)
            buf[:, :, :self.nao] = ao[:, :, :self.nao]
            ao = buf
        self._grid_keep = [ao, weights]
        _lib.check(self.lib.xtd_set_grid(self._h, _ptr(ao), nvar, ng, ao.stride(1), ao.stride(0), _ptr(weights)), "xtd_set_grid")

    def set_fxc(self, kind: str, fxc):
        if kind != "none":
            assert fxc.is_contiguous()
            if self.plan.xc_scale != 1.0:       # the grid term is linear in the kernel table (Z-vector plans: hermi = 1 densities)
                fxc = fxc * float(self.plan.xc_scale)
            # the ALDA0 kernel f[ng] is read on every call; the UKS / multicollinear tensors only by grid_commit
            (self._keep if kind == "alda0" else self._grid_keep).append(fxc)
        _lib.check(self.lib.xtd_set_fxc(self._h, _KIND[kind], _ptr(fxc) if kind != "none" else None), "xtd_set_fxc")

    def grid_commit(self):
        """AO values -> occupied / virtual MO values on the grid (once per solve).  Afterwards the AO array, the weights
        and the UKS / multicollinear kernel tensor are released: the engine keeps only MO values and its kernel table."""
        self._set_stream()
        _lib.check(self.lib.xtd_grid_commit(self._h), "xtd_grid_commit")
        self._grid_keep = []

    # ---- finalize -----------------------------------------------------------------------------------
    def finalize(self, max_nvec: int = 40):
        plan = self.plan
        self._set_stream()
        for lg in plan.local_gemms:
            m = np.ascontiguousarray(lg.mat, dtype=np.float64)
            dc, r0, nr, c0, ncol = lg.dst
            sc, sr0, sc0 = lg.src
            side = {"R": _lib.XTD_SIDE_RIGHT, "L": _lib.XTD_SIDE_LEFT, "LT": _lib.XTD_SIDE_LEFT_T, "RT": _lib.XTD_SIDE_RIGHT_T}[lg.side]
            _lib.check(self.lib.xtd_add_local_gemm(self._h, side, dc, r0, nr, c0, ncol, sc, sr0, sc0, _np_ptr(m), m.shape[0], m.shape[1],
                                                   float(lg.alpha)), "xtd_add_local_gemm")
        for r1 in plan.rank1s:
            u = np.ascontiguousarray(r1.u, dtype=np.float64)
            v = np.ascontiguousarray(r1.v, dtype=np.float64)
            _lib.check(self.lib.xtd_add_rank1(self._h, r1.dst_ch, _np_ptr(u), r1.src_ch, _np_ptr(v)), "xtd_add_rank1")
        for dg in plan.diags:
            d = np.ascontiguousarray(dg.d, dtype=np.float64)
            _lib.check(self.lib.xtd_add_diag(self._h, dg.ch, _np_ptr(d)), "xtd_add_diag")
        # layout maps
        lds, offs = [], []
        for ci in range(len(plan.channels)):
            base, vs, ld = C.c_long(), C.c_long(), C.c_long()
            _lib.check(self.lib.xtd_channel_layout(self._h, ci, 1, C.byref(base), C.byref(vs), C.byref(ld)), "xtd_channel_layout")
            lds.append(ld.value)
            offs.append(0)                      # scatter offsets are channel-local; the engine adds the channel base
            g = plan.gather_map(ci)
            _lib.check(self.lib.xtd_set_gather(self._h, ci, _np_ptr(g.indptr), _np_ptr(g.cols), _np_ptr(g.vals), len(g.cols)),
                       "xtd_set_gather")
        sm = plan.scatter_map(offs, lds)
        ent = plan.layout_entries
        order = np.argsort(ent[:, 0], kind="stable")
        chans = np.ascontiguousarray(ent[order, 1].astype(np.int8))
        _lib.check(self.lib.xtd_set_scatter(self._h, plan.ext_dim, _np_ptr(sm.indptr), _np_ptr(sm.cols), _np_ptr(chans), _np_ptr(sm.vals),
                                            len(sm.cols)), "xtd_set_scatter")
        _lib.check(self.lib.xtd_finalize(self._h, int(max_nvec)), "xtd_finalize")
        self._grid_keep = []                    # xtd_finalize implies the grid commit
        self.max_nvec = int(max_nvec)
        self.finalized = True

    @classmethod
    def from_problem(cls, plan: Plan, p: ProblemData, *, max_nvec: int = 40, workspace_bytes: int = 2 << 30, device=None,
                     reducer: Optional[SigmaReducer] = None, rank: int = 0, world: int = 1, df_chunk: int = 64,
                     exchange_slices: Optional[int] = None, plan_builder=None) -> "SigmaEngine":
        """Upload a host ProblemData; with world > 1 this rank keeps only its aux block and grid batch.

        `plan_builder(p) -> Plan`: for a ROKS problem WITHOUT ROHF-form Fock matrices (`p.fock_hf is None`) the engine computes
        their spin difference K[D_open] on the device while the tensor streams in, stores it as `p.fock_hf = [0, K]` (only the
        difference enters the sigma build) and compiles the final plan with `plan_builder` before the local terms are uploaded;
        `plan` then only has to carry the channels and exchange / Coulomb declarations (built from a zero placeholder)."""
        import torch
        need_kopen = bool(p.restricted and p.fock_hf is None and plan_builder is not None)
        if need_kopen:
            p.fock_hf = np.zeros((2, p.nmo, p.nmo))
            plan = plan_builder(p)
        eng = cls(plan, p.nao, p.mo_coeff, workspace_bytes=workspace_bytes, device=device, reducer=reducer, exchange_slices=exchange_slices)
        g0, g1 = split_range(p.ng, rank, world) if plan.xc_kind != "none" else (0, 0)
        if g1 > g0:                             # a rank whose grid batch is empty simply has no grid term
            ld = _pad16(p.nao)
            ao = torch.zeros((p.nvar, g1 - g0, ld), dtype=torch.float64, device=eng.device)
            ao[:, :, :p.nao] = torch.from_numpy(np.ascontiguousarray(p.ao[:, g0:g1])).to(eng.device)
            w = torch.from_numpy(np.ascontiguousarray(p.weights[g0:g1])).to(eng.device)
            eng.set_grid(ao, w)
            if plan.xc_kind in ("uks", "uks_tau"):
                f = torch.from_numpy(np.ascontiguousarray(p.fxc_uks[..., g0:g1])).to(eng.device)
            elif plan.xc_kind == "alda0":
                f = torch.from_numpy(np.ascontiguousarray(p.fxc_alda0[g0:g1])).to(eng.device)
            else:
                f = torch.from_numpy(np.ascontiguousarray(p.fxc_mcol[..., g0:g1])).to(eng.device)
            eng.set_fxc(plan.xc_kind, f)
            del ao, w, f
            eng.grid_commit()                   # AO values are dropped before the tensor streams in
            torch.cuda.empty_cache()
        if need_kopen:
            if 0 not in eng.tensors_used:
                raise _lib.XtdError("the ROHF-form Fock difference needs the density-fitting tensor, but this plan streams none")
            eng.set_open_orbitals(0, np.arange(p.nc, p.nc + p.no))
        for t in eng.tensors_used:
            full = p.cderi if t == 0 else p.cderi_lr
            if full is None:                    # PySCF's packed storage: streamed block by block, never unpacked on the host
                eng.load_cderi_packed(t, p.cderi_packed if t == 0 else p.cderi_lr_packed, p.naux_packed, rank, world, chunk=df_chunk)
                continue
            p0, p1 = split_range(full.shape[0], rank, world)
            eng.load_cderi(t, full[p0:p1], chunk=df_chunk)
        if need_kopen:
            p.fock_hf = np.stack([np.zeros((p.nmo, p.nmo)), eng.kopen()])
            eng.plan = plan_builder(p)          # same channels / exchange declarations, local terms with the computed couplings
        eng.finalize(max_nvec)
        return eng

    # ---- preconditioner diagonal ----------------------------------------------------------------------
    def jblock_diag(self, jb: int) -> np.ndarray:
        torch = self.torch
        blk = self.plan.j_blocks[jb]
        out = torch.zeros(blk.nr * blk.nc, dtype=torch.float64, device=self.device)
        self._set_stream()
        _lib.check(self.lib.xtd_jblock_diag(self._h, jb, _ptr(out)), "xtd_jblock_diag")
        if self.reducer is not None:
            self.reducer.allreduce_(out)
        return out.cpu().numpy().reshape(blk.nr, blk.nc)

    def hdiag(self) -> np.ndarray:
        plan = self.plan
        if plan.hdiag_needs_jdiag is None:
            return np.asarray(plan.hdiag)
        co_j = ov_j = None
        if plan.hdiag_needs_jdiag["pending"] is not None:
            co_j, ov_j = self.jblock_diag(0), self.jblock_diag(1)
        return finish_xsf_hdiag(plan, co_j, ov_j)

    # ---- the operator -----------------------------------------------------------------------------------
    def sigma(self, z, out=None):
        """z: torch cuda fp64 [nvec, dim] (contiguous).  Returns torch cuda [nvec, dim]."""
        torch = self.torch
        assert self.finalized
        assert z.is_cuda and z.dtype == torch.float64 and z.dim() == 2 and z.shape[1] == self.ext_dim and z.is_contiguous()
        nvec = z.shape[0]
        if out is None:
            out = torch.empty_like(z)
        self._set_stream()
        for x0 in range(0, nvec, self.max_nvec):
            x1 = min(nvec, x0 + self.max_nvec)
            zz, oo = z[x0:x1], out[x0:x1]
            if self.reducer is None or not self.reducer.enabled:
                _lib.check(self.lib.xtd_sigma(self._h, x1 - x0, _ptr(zz), _ptr(oo)), "xtd_sigma")
            else:
                _lib.check(self.lib.xtd_sigma_partial(self._h, x1 - x0, _ptr(zz)), "xtd_sigma_partial")
                ptr, n = C.c_void_p(), C.c_long()
                _lib.check(self.lib.xtd_partial_buffer(self._h, x1 - x0, C.byref(ptr), C.byref(n)), "xtd_partial_buffer")
                part = _as_tensor(torch, ptr.value, n.value, self.device)
                ev = self._ar_events()
                ev[0].record()
                self.reducer.allreduce_(part)          # one all-reduce(sum, fp64) of the MO-space partial per call
                ev[1].record()
                self._ar_pending.append(ev)
                _lib.check(self.lib.xtd_sigma_finish(self._h, x1 - x0, _ptr(oo)), "xtd_sigma_finish")
        return out

    def block_response(self, dens: np.ndarray, coef, x: Optional[np.ndarray] = None):
        """Responses of symmetric MO-block densities on the resident blocks (xtd_block_response; the plan needs `block_response`).
        dens: per channel [Doo (no x no) | Dvv (nv x nv) | Dov (no x nv)] flattened on the channel's internal positions;
        coef = (J, K tensor 0, K tensor 1, f_xc, K[X]).  Returns (per channel [Voo | Vov] flattened, K[X] on (channel-1 occ + vir) x
        (channel-0 occ + vir) or None), summed over the ranks.

        Several densities at once: dens[k, n] and x[k, no_1, nv_0] (or [k, no_1 * nv_0]) with one coef; the outputs gain the same
        leading axis.  One xtd_block_response_batch call reads the resident blocks once per pass for all k densities, and with several
        ranks the whole batch is all-reduced once."""
        torch = self.torch
        assert self.finalized and self.plan.block_response
        chs = self.plan.channels
        nin = sum(c.no * c.no + c.nv * c.nv + c.no * c.nv for c in chs)
        nout = sum(c.no * c.no + c.no * c.nv for c in chs)
        nxin, nxout = chs[1].no * chs[0].nv, (chs[1].no + chs[1].nv) * (chs[0].no + chs[0].nv)
        dens = np.ascontiguousarray(dens, dtype=np.float64)
        batched = dens.ndim == 2
        if dens.ndim not in (1, 2) or dens.shape[-1] != nin:
            raise ValueError(f"block_response: dens must be [{nin}] or [k, {nin}], got {dens.shape}")
        k = dens.shape[0] if batched else 1
        if k == 0:
            raise ValueError("block_response: empty batch")
        d = torch.from_numpy(dens.ravel()).to(self.device)
        c = np.ascontiguousarray(coef, dtype=np.float64)
        assert c.shape == (5,)
        # one buffer for the responses and K[X]: a single all-reduce per call
        res = torch.empty(k * (nout + (nxout if x is not None else 0)), dtype=torch.float64, device=self.device)
        out, xo = res[:k * nout], None
        xd = None
        if x is not None:
            xh = np.ascontiguousarray(x, dtype=np.float64)
            if xh.size != k * nxin or (batched and xh.shape[0] != k):
                raise ValueError(f"block_response: x must hold {k} blocks of {chs[1].no} x {chs[0].nv}, got {xh.shape}")
            xd = torch.from_numpy(xh.ravel()).to(self.device)
            xo = res[k * nout:]
        self._set_stream()
        xp, xop = (_ptr(xd), _ptr(xo)) if xd is not None else (None, None)
        if batched:
            _lib.check(self.lib.xtd_block_response_batch(self._h, k, _ptr(d), _ptr(out), _np_ptr(c), xp, xop), "xtd_block_response_batch")
        else:
            _lib.check(self.lib.xtd_block_response(self._h, _ptr(d), _ptr(out), _np_ptr(c), xp, xop), "xtd_block_response")
        if self.reducer is not None and self.reducer.enabled:
            self.reducer.allreduce_(res)
        res = res.cpu().numpy()
        out, xo = res[:k * nout], (res[k * nout:] if x is not None else None)
        if batched:
            return out.reshape(k, nout), (xo.reshape(k, nxout) if xo is not None else None)
        return out, xo

    def last_density_batches(self) -> int:
        """Passes over the densities the last batched block_response made (more than one when the workspace could not hold them all)."""
        n = C.c_long()
        _lib.check(self.lib.xtd_last_density_batches(self._h, C.byref(n)), "xtd_last_density_batches")
        return n.value

    def sigma_host(self, z: np.ndarray) -> np.ndarray:
        """Reference-facing entry with HOST vectors: H2D + sigma + D2H inside the C-ABI call (single rank)."""
        z = np.ascontiguousarray(z, dtype=np.float64)
        if z.ndim == 1:
            z = z[None]
        out = np.empty_like(z)
        if self.reducer is not None and self.reducer.enabled:
            t = self.torch.from_numpy(z).to(self.device)
            return self.sigma(t).cpu().numpy()
        self._set_stream()
        for x0 in range(0, z.shape[0], self.max_nvec):
            x1 = min(z.shape[0], x0 + self.max_nvec)
            _lib.check(self.lib.xtd_sigma_host(self._h, x1 - x0, _np_ptr(z[x0:x1]), _np_ptr(out[x0:x1])), "xtd_sigma_host")
        return out

    def as_vind(self):
        """`vind(zs)` with the reference's contract (XTDA.py:615, SF_TDA.py:224): list / array in, new array out."""
        def vind(zs):
            return self.sigma_host(np.asarray(zs, dtype=np.float64).reshape(-1, self.ext_dim))
        return vind

    def _ar_events(self):
        """A pair of CUDA events around the all-reduce of one call (device time of the collective as this rank sees it,
        waiting for the slowest rank included)."""
        if not hasattr(self, "_ar_pool"):
            self._ar_pool, self._ar_pending = [], []
        if self._ar_pool:
            return self._ar_pool.pop()
        return (self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True))

    def stats(self) -> dict:
        """Per-phase device times (ms) and GEMM flops of the LAST sigma call; `allreduce` = the NCCL all-reduce of every
        partial-sigma block since the previous stats() call."""
        st = _lib.XtdStats()
        _lib.check(self.lib.xtd_get_stats(self._h, C.byref(st)), "xtd_get_stats")
        ms = {n: st.ms[i] for i, n in enumerate(_lib.T_NAMES)}
        ar = 0.0
        for ev in getattr(self, "_ar_pending", []):
            ar += ev[0].elapsed_time(ev[1])         # xtd_get_stats synchronised the stream
            self._ar_pool.append(ev)
        if hasattr(self, "_ar_pending"):
            self._ar_pending = []
        ms["allreduce"] = ar
        return dict(flops_gemm=st.flops_gemm, launches=int(st.launches), ms=ms, flops={n: st.flops[i] for i, n in enumerate(_lib.T_NAMES)})

    def last_chunks(self):
        """(aux chunks, grid chunks) the last eager sigma call looped over."""
        a, g = C.c_long(), C.c_long()
        _lib.check(self.lib.xtd_last_chunks(self._h, C.byref(a), C.byref(g)), "xtd_last_chunks")
        return a.value, g.value

    def reset_stats(self):
        _lib.check(self.lib.xtd_reset_stats(self._h), "xtd_reset_stats")


def _as_tensor(torch, ptr: int, n: int, device):
    """Wrap a raw device pointer (owned by the engine's workspace) as a torch tensor, without copying."""
    class _Holder:
        pass
    h = _Holder()
    h.__cuda_array_interface__ = dict(shape=(n,), typestr="<f8", data=(ptr, False), version=3, strides=None)
    return torch.as_tensor(h, device=device)
