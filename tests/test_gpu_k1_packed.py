"""The fused half-transform on its packed Loo image: the rows (P, i) of a group of aux functions share 128-row tiles, and CTA pairs
share the Loo stage by cluster multicast.  The emulated engine (6 digit planes) is compared with the FP64 engine on the same problem:
occupied counts just below and just above a multiple of 128 (row tiles that straddle aux functions, a ragged last group, several aux
chunks), an odd count of (vector, column tile) items (the masked partner of the last pair), a block-weighted term with two occupied
row blocks, and aux shards.  Needs a B200."""
import ctypes as C

import numpy as np
import pytest

from xtddft_b200 import plan as planmod
from xtddft_b200.synth import make_problem

pytestmark = pytest.mark.gpu

TOL = 1e-11     # the emulated-path tolerance of tests/test_gpu_ozaki.py at 6-7 planes


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _rel(got, ref):
    return float(np.abs(got - ref).max() / max(1.0, np.abs(ref).max()))


def _sigma(torch, plan, p, z, slices, **kw):
    from xtddft_b200.engine import SigmaEngine
    eng = SigmaEngine.from_problem(plan, p, workspace_bytes=512 << 20, max_nvec=4, exchange_slices=slices, **kw)
    got = eng.sigma(torch.from_numpy(z).cuda()).cpu().numpy()
    info = (eng.last_chunks()[0], eng.stats()["ms"])
    eng.close()
    return got, info


# nc + no occupied rows per aux function: 127 (4 x 127 = 508 rows in 4 tiles) and 129 (4 x 129 = 516 rows in 5 tiles)
@pytest.mark.parametrize("nc", [125, 127])
@pytest.mark.parametrize("nv,nvec", [(150, 3), (200, 4)])
def test_k1_packed_rows_against_fp64(torch_cuda, monkeypatch, nc, nv, nvec):
    """SF-TDA, 23 aux functions in chunks of 4 (the last group holds 3), occupied count just below / above 128.  nv = 150 with 3
    vectors: 3 column tiles x 3 vectors is odd, so the second CTA of the last pair of every row tile is masked."""
    monkeypatch.setenv("XTD_CHUNK_AUX", "5")
    p = make_problem(nc + 2 + nv, nc, 2, nv, 23, 200, xctype="LDA", hyb=0.5, seed=500 + nc)
    plan = planmod.build_sf_plan(p, isf=-1, method=0)
    z = np.random.default_rng(11).standard_normal((nvec, plan.ext_dim))
    ref, _ = _sigma(torch_cuda, plan, p, z, 0)
    got, (chunks, ms) = _sigma(torch_cuda, plan, p, z, 6)
    assert ms["k1"] > 0, "the fused half-transform did not run"
    assert chunks == 6, chunks
    assert _rel(got, ref) < TOL


@pytest.mark.parametrize("nc,no", [(140, 3), (60, 4)])
def test_k1_packed_two_row_blocks_against_fp64(torch_cuda, monkeypatch, nc, no):
    """XSF-TDA Delta A: a block-weighted exchange term with two occupied row blocks (closed and open rows), one half-transform pass
    per block over its own packed rows, several aux chunks."""
    monkeypatch.setenv("XTD_CHUNK_AUX", "8")
    nv = 150
    p = make_problem(nc + no + nv, nc, no, nv, 19, 200, xctype="LDA", hyb=0.3, seed=520 + no)
    plan = planmod.build_sf_plan(p, isf=-1, method=0, sa=3, layout=planmod.LAYOUT_BLOCK, remove=True, foo=0.8, fglobal=0.7,
                                 hdiag_kind="xsf")
    z = np.random.default_rng(12).standard_normal((3, plan.ext_dim))
    ref, _ = _sigma(torch_cuda, plan, p, z, 0, df_chunk=12)
    got, (chunks, ms) = _sigma(torch_cuda, plan, p, z, 6, df_chunk=12)
    assert ms["k1"] > 0, "the fused half-transform did not run"
    assert chunks == 3, chunks
    assert _rel(got, ref) < TOL


def test_k1_packed_shards_against_fp64(torch_cuda):
    """Three aux shards of 11 / 11 / 11 functions (each shard's last group is ragged) whose partial buffers add up to the FP64 result."""
    from xtddft_b200 import _lib
    from xtddft_b200.engine import SigmaEngine, _as_tensor
    torch = torch_cuda
    p = make_problem(160, 129, 2, 29, 33, 100, xctype="LDA", hyb=0.5, seed=530)
    plan = planmod.build_sf_plan(p, isf=-1, method=0)
    z = np.random.default_rng(13).standard_normal((3, plan.ext_dim))
    ref, _ = _sigma(torch, plan, p, z, 0)
    zt = torch.from_numpy(z).cuda()
    acc = None
    for r in range(3):
        eng = SigmaEngine.from_problem(plan, p, workspace_bytes=128 << 20, max_nvec=4, rank=r, world=3, exchange_slices=6)
        _lib.check(eng.lib.xtd_sigma_partial(eng._h, 3, C.c_void_p(zt.data_ptr())), "partial")
        ptr, n = C.c_void_p(), C.c_long()
        _lib.check(eng.lib.xtd_partial_buffer(eng._h, 3, C.byref(ptr), C.byref(n)), "buffer")
        part = _as_tensor(torch, ptr.value, n.value, eng.device).clone()
        acc = part if acc is None else acc + part
        if r == 2:
            _as_tensor(torch, ptr.value, n.value, eng.device).copy_(acc)
            out = torch.empty_like(zt)
            _lib.check(eng.lib.xtd_sigma_finish(eng._h, 3, C.c_void_p(out.data_ptr())), "finish")
            assert _rel(out.cpu().numpy(), ref) < TOL
        eng.close()
