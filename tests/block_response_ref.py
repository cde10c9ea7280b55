"""NumPy restatement of `xtd_block_response` (csrc/xtd_api.cu) on the engine's index sets and with its factorisation: the MO blocks
Loo / Lov / Lvv of every channel, the exchange through A = Loo Doo + Lov Dov^T and B = Loo Dov + Lov Dvv, the mixed-spin K[X] through
U = Loo_1 X and V = Lov_1^T X, the fitted Coulomb density, and the grid term through Wo / Wv and the weighted occupied values Bo.
Test infrastructure: the CPU suite feeds it to `zvector.block_callables` to check the block bookkeeping against the reference's own
right-hand sides and W matrices."""
import numpy as np


def _cols(c, idx):
    out = np.zeros((c.shape[0], len(idx)))
    idx = np.asarray(idx)
    out[:, idx >= 0] = c[:, idx[idx >= 0]]
    return out


def block_response_numpy(p, plan, dens, coef, x=None):
    chs = plan.channels
    cj, ck0, ck1, cxc, cx = [float(c) for c in coef]
    co = [_cols(p.mo_coeff[ch.spin_o], ch.occ_idx) for ch in chs]
    cv = [_cols(p.mo_coeff[ch.spin_v], ch.vir_idx) for ch in chs]
    D, off = [], 0
    for ch in chs:
        no, nv = ch.no, ch.nv
        doo = dens[off:off + no * no].reshape(no, no); off += no * no
        dvv = dens[off:off + nv * nv].reshape(nv, nv); off += nv * nv
        dov = dens[off:off + no * nv].reshape(no, nv); off += no * nv
        D.append((doo, dvv, dov))
    O = [[np.zeros((ch.no, ch.no)), np.zeros((ch.no, ch.nv))] for ch in chs]
    xo = None
    es = lambda *a: np.einsum(*a, optimize=True)
    for t, ck in ((0, ck0), (1, ck1)):
        cderi = p.cderi if t == 0 else p.cderi_lr
        doj, dox = t == 0 and cj != 0.0, t == 0 and x is not None and cx != 0.0
        if cderi is None or not (doj or ck != 0.0 or dox):
            continue
        L = [(es("Pmn,mi,nj->Pij", cderi, co[c], co[c]), es("Pmn,mi,nj->Pij", cderi, co[c], cv[c]), es("Pmn,mi,nj->Pij", cderi, cv[c], cv[c]))
             for c in range(2)]
        if doj:
            rho = sum(es("Pij,ij->P", L[c][0], D[c][0]) + es("Pij,ij->P", L[c][2], D[c][1]) + 2 * es("Pij,ij->P", L[c][1], D[c][2]) for c in range(2))
            for c in range(2):
                O[c][0] += cj * es("P,Pij->ij", rho, L[c][0])
                O[c][1] += cj * es("P,Pij->ij", rho, L[c][1])
        if ck != 0.0:
            for c in range(2):
                loo, lov, lvv = L[c]
                doo, dvv, dov = D[c]
                A = loo @ doo + lov @ dov.T
                B = loo @ dov + lov @ dvv
                O[c][0] += ck * (es("Pij,Pjk->ik", A, loo) + es("Pia,Pka->ik", B, lov))
                O[c][1] += ck * (es("Pij,Pja->ia", A, lov) + es("Pib,Pba->ia", B, lvv))
        if dox:
            xb = np.asarray(x).reshape(chs[1].no, chs[0].nv)
            U = L[1][0] @ xb
            V = L[1][1].transpose(0, 2, 1) @ xb
            xo = cx * np.block([[es("Pib,Pjb->ij", U, L[0][1]), es("Pib,Pba->ia", U, L[0][2])],
                                [es("Pib,Pjb->ij", V, L[0][1]), es("Pib,Pba->ia", V, L[0][2])]])
    if cxc != 0.0 and plan.xc_kind != "none" and p.ng > 0:
        fxc = p.fxc_uks * plan.xc_scale
        tau = fxc.shape[1] == 5
        nvar = p.ao.shape[0]
        phi = [es("cgm,mi->cgi", p.ao, co[c]) for c in range(2)]
        phiv = [es("cgm,ma->cga", p.ao, cv[c]) for c in range(2)]
        rho = []
        for c in range(2):
            doo, dvv, dov = D[c]
            wo = phi[c] @ doo + phiv[c] @ dov.T
            wv = phiv[c] @ dvv + phi[c] @ dov
            r = [es("gi,gi->g", phi[c][0], wo[0]) + es("ga,ga->g", phiv[c][0], wv[0])]
            r += [2 * (es("gi,gi->g", phi[c][k], wo[0]) + es("ga,ga->g", phiv[c][k], wv[0])) for k in range(1, nvar)]
            if tau:
                r.append(0.5 * sum(es("gi,gi->g", phi[c][k], wo[k]) + es("ga,ga->g", phiv[c][k], wv[k]) for k in range(1, 4)))
            rho.append(np.stack(r))
        wvs = es("axg,axbyg->byg", np.stack(rho), fxc) * p.weights
        for c in range(2):
            w = wvs[c]
            bo = np.empty_like(phi[c])
            bo[0] = w[0][:, None] * phi[c][0] + sum(w[k][:, None] * phi[c][k] for k in range(1, nvar))
            for k in range(1, nvar):
                bo[k] = w[k][:, None] * phi[c][0] + (0.5 * w[4][:, None] * phi[c][k] if tau else 0.0)
            O[c][0] += cxc * es("cgi,cgj->ij", bo, phi[c])
            O[c][1] += cxc * es("cgi,cga->ia", bo, phiv[c])
    out = np.concatenate([np.concatenate([O[c][0].ravel(), O[c][1].ravel()]) for c in range(2)])
    return out, (xo.ravel() if xo is not None else None)
