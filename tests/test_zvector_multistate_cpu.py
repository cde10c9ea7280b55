"""Several Z-vector states at once, on the CPU: the block Galerkin solver (`solve_linear_block`) on NumPy vectors against
numpy.linalg.solve and `solve_linear`, and the batched block callables fed by a loop over the NumPy restatement of
`xtd_block_response` against the five `zvector_*` fixtures, each fixture state inside a batch of seeded states."""
import os

import numpy as np
import pytest

from block_response_ref import block_response_numpy
from numpy_vectors import NumpyVectors
from test_zvector_blocks_cpu import TAGS
from xtddft_b200 import plan as planmod
from xtddft_b200.synth import make_problem
from xtddft_b200.zvector import (assemble_rhs, assemble_w, block_callables_many, per_state_batched, rhs_intermediates, solve_linear,
                                 solve_linear_block)


def _rel(a, b):
    return float(np.abs(a - b).max() / max(1.0, np.abs(b).max()))


def _operator(n, symmetric, seed):
    rng = np.random.default_rng(seed)
    a = rng.standard_normal((n, n)) * 0.1
    if symmetric:
        a = a + a.T
    a += np.diag(np.linspace(1.0, 4.0, n))
    return a


class _Counted:
    def __init__(self, a, max_nvec):
        self.a, self.max_nvec, self.calls, self.widths = a, max_nvec, 0, []

    def __call__(self, x):
        assert 1 <= x.shape[0] <= self.max_nvec
        self.calls += 1
        self.widths.append(x.shape[0])
        return x @ self.a.T


@pytest.mark.parametrize("symmetric", [True, False])
@pytest.mark.parametrize("k,max_nvec", [(3, 4), (6, 4), (5, 2)])
def test_block_solve_against_numpy(symmetric, k, max_nvec):
    n = 60
    a = _operator(n, symmetric, 5 + k)
    b = np.random.default_rng(k).standard_normal((k, n))
    aop = _Counted(a, max_nvec)
    x, conv, cycles, res, calls = solve_linear_block(aop, b, np.diag(a), tol=1e-11, max_cycle=n, max_nvec=max_nvec,
                                                     backend=NumpyVectors(n))
    ref = np.linalg.solve(a, b.T).T
    assert conv.all() and (res < 1e-11).all()
    assert np.abs(x - ref).max() < 1e-9 * np.abs(ref).max()
    assert calls == aop.calls and (cycles <= calls).all()
    for i in range(k):
        assert np.linalg.norm(a @ x[i] - b[i]) < 1e-10


@pytest.mark.parametrize("symmetric", [True, False])
def test_one_system_matches_solve_linear(symmetric):
    n = 40
    a = _operator(n, symmetric, 11)
    b = np.random.default_rng(3).standard_normal(n)
    hd = np.diag(a)
    x1, c1, k1, r1 = solve_linear(lambda v: v @ a.T, b, hd, tol=1e-12, max_cycle=n, backend=NumpyVectors(n))
    xb, cb, kb, rb, calls = solve_linear_block(lambda v: v @ a.T, b[None], hd, tol=1e-12, max_cycle=n, backend=NumpyVectors(n))
    assert cb[0] == c1 and kb[0] == k1 == calls
    assert abs(rb[0] - r1) <= 1e-14 * max(1.0, r1) + 1e-18
    assert np.abs(xb[0] - x1).max() <= 1e-12 * np.abs(x1).max()


def test_zero_rhs_converges_at_once():
    n = 30
    a = _operator(n, False, 2)
    b = np.random.default_rng(4).standard_normal((3, n))
    b[1] = 0.0
    x, conv, cycles, res, calls = solve_linear_block(lambda v: v @ a.T, b, np.diag(a), tol=1e-11, max_cycle=n, backend=NumpyVectors(n))
    assert conv.all() and cycles[1] == 0 and res[1] == 0.0
    assert not x[1].any()
    assert np.abs(x[[0, 2]] - np.linalg.solve(a, b[[0, 2]].T).T).max() < 1e-9


def test_identical_rhs_drop_dependent_directions():
    n = 30
    a = _operator(n, True, 6)
    b0 = np.random.default_rng(5).standard_normal(n)
    b = np.stack([b0, b0, 2.0 * b0])
    aop = _Counted(a, 4)
    x, conv, cycles, res, calls = solve_linear_block(aop, b, np.diag(a), tol=1e-11, max_cycle=n, backend=NumpyVectors(n))
    assert conv.all()
    assert aop.widths[0] == 1          # the copies' first directions fall below lindep: the first call carries one vector
    ref = np.linalg.solve(a, b0)
    for i, s in enumerate((1.0, 1.0, 2.0)):
        assert np.abs(x[i] - s * ref).max() < 1e-9 * max(1.0, np.abs(ref).max())


def _fixture(golden_dir, tag):
    d = np.load(os.path.join(golden_dir, f"zvector_{tag}.npz"), allow_pickle=False)
    nc, no, nv, naux, ng, seed, restricted = [int(x) for x in d["params"]]
    p = make_problem(nc + no + nv, nc, no, nv, naux, ng, xctype=str(d["xctype"]), hyb=float(d["hyb"]), restricted=bool(restricted),
                     seed=seed)
    return d, p


def _ref_batch(p, plan, calls):
    def apply(dens, coef, x):
        assert dens.ndim == 2 and (x is None or len(x) == len(dens))
        calls.append(len(dens))
        outs = [block_response_numpy(p, plan, dens[i], coef, None if x is None else x[i]) for i in range(len(dens))]
        return np.stack([o[0] for o in outs]), (np.stack([o[1] for o in outs]) if x is not None else None)
    return apply


@pytest.mark.parametrize("tag", TAGS)
def test_batched_callables_reproduce_fixtures(golden_dir, tag):
    """The fixture state in the middle of a batch of three: its right-hand side and W matrix match the goldens; every batched
    callable is called once for the whole batch."""
    d, p = _fixture(golden_dir, tag)
    plan = planmod.build_zvector_plan(p)
    rng = np.random.default_rng(17)
    V = np.stack([rng.standard_normal((p.nc, p.nv)), d["amp"].reshape(p.nc, p.nv), rng.standard_normal((p.nc, p.nv))])
    Z = np.stack([rng.standard_normal(plan.ext_dim), d["z"], rng.standard_normal(plan.ext_dim)])
    calls = []
    resp, sfx, full = block_callables_many(p, plan, _ref_batch(p, plan, calls))
    inters = per_state_batched(3, lambda i, r, x: rhs_intermediates(p, V[i], r, x), resp, sfx)
    assert calls == [3] * (2 if p.hyb != 0.0 else 1)
    rhs = np.stack([assemble_rhs(p, V[i], None, None, inter=it) for i, it in enumerate(inters)])
    w = per_state_batched(3, lambda i, f: assemble_w(p, Z[i], inters[i], f), full)
    assert calls[-1] == 3 and len(calls) == (3 if p.hyb != 0.0 else 2)
    assert _rel(rhs[1], d["rhs"]) < 1e-12
    assert _rel(w[1], d["im0"]) < 1e-12
    # the other members equal their single-state results
    from xtddft_b200.zvector import block_callables
    r1, s1, f1 = block_callables(p, plan, lambda dd, c, x: block_response_numpy(p, plan, dd, c, x))
    for i in (0, 2):
        it = rhs_intermediates(p, V[i], r1, s1)
        assert _rel(rhs[i], assemble_rhs(p, V[i], None, None, inter=it)) < 1e-13
        assert _rel(w[i], assemble_w(p, Z[i], it, f1)) < 1e-13
