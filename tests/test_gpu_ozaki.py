"""FP64 contraction emulated on the INT8 tensor cores (tcgen05.mma kind::i8 + TMEM, csrc/ozaki.cuh) against an fp64
reference of the same contraction (numpy on the host: the oracle for a floating-point kernel is the plain fp64 product).
Error model: each operand row is cut into S radix-256 digit planes below a power-of-two row scale, products with i + j >= S
are dropped, so |C - C_ref| <~ (S + 2) 2^(7 - 8 S) * K * rowmax(a) rowmax(b) -- with S >= 7 that is the fp64 rounding level.
Needs a B200."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _ozaki(torch, a, b, slices, group=0, alpha=1.0, c0=None):
    """a [nq, M, K], b [nq, N, K] (numpy) -> C [M, N] through xtd_ozaki_gemm with padded leading dimensions."""
    from xtddft_b200 import _lib
    lib = _lib.load()
    nq, m, k = a.shape
    n = b.shape[1]
    ld = (k + 15) // 16 * 16
    ad = torch.full((nq, m, ld), 7.0, dtype=torch.float64, device="cuda")      # garbage in the padding: must be ignored
    bd = torch.full((nq, n, ld), -3.0, dtype=torch.float64, device="cuda")
    ad[:, :, :k] = torch.from_numpy(a).cuda()
    bd[:, :, :k] = torch.from_numpy(b).cuda()
    ldc = (n + 1) // 2 * 2
    cd = torch.zeros((m, ldc), dtype=torch.float64, device="cuda")
    if c0 is not None:
        cd[:, :n] = torch.from_numpy(c0).cuda()
    ms = (C.c_double * 3)()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(lib.xtd_ozaki_gemm(st, m, n, k, nq, slices, group, C.c_void_p(ad.data_ptr()), ld, m * ld, C.c_void_p(bd.data_ptr()), ld, n * ld,
                                  C.c_void_p(cd.data_ptr()), ldc, alpha, 1 if c0 is not None else 0, ms), "xtd_ozaki_gemm")
    return cd[:, :n].cpu().numpy(), list(ms)


def _ref(a, b):
    return np.einsum("qmk,qnk->mn", a, b, optimize=True)


@pytest.mark.parametrize("m,n,k,nq", [(128, 64, 32, 1), (100, 50, 70, 3), (300, 200, 129, 5), (17, 9, 5, 2), (257, 130, 64, 20)])
def test_ozaki_small_exact_level(torch_cuda, m, n, k, nq):
    """8 planes: 64 bits below the row scale -> agreement at the fp64 rounding level; ragged M, N, K and several q-slices."""
    rng = np.random.default_rng(m + n + k)
    a = rng.standard_normal((nq, m, k))
    b = rng.standard_normal((nq, n, k))
    c, _ = _ozaki(torch_cuda, a, b, 8)
    ref = _ref(a, b)
    bound = np.einsum("qmk,qnk->mn", np.abs(a), np.abs(b)).max()
    assert np.abs(c - ref).max() <= 1e-13 * bound


def test_ozaki_integer_inputs_are_exact(torch_cuda):
    """Small integers are represented exactly by the first two digits: the int8 pipeline must reproduce the product bit
    for bit (catches any descriptor / layout / level-weight mistake without tolerance)."""
    rng = np.random.default_rng(5)
    a = rng.integers(-50, 51, (4, 256, 96)).astype(np.float64)
    b = rng.integers(-50, 51, (4, 128, 96)).astype(np.float64)
    for s in (3, 5, 8):
        c, _ = _ozaki(torch_cuda, a, b, s)
        assert np.array_equal(c, _ref(a, b)), s


@pytest.mark.parametrize("slices", [3, 4, 5, 6, 7, 8])
def test_ozaki_error_vs_slices(torch_cuda, slices):
    """Truncation error drops by 2^-8 per plane; rows with a wide dynamic range (1e-6 .. 1) inside one scale group."""
    rng = np.random.default_rng(9)
    nq, m, n, k = 6, 200, 150, 300
    a = rng.standard_normal((nq, m, k)) * 10.0 ** rng.uniform(-6, 0, (nq, m, k))
    b = rng.standard_normal((nq, n, k)) * 10.0 ** rng.uniform(-6, 0, (nq, n, k))
    c, _ = _ozaki(torch_cuda, a, b, slices, group=2)
    ref = _ref(a, b)
    # row / column maxima over a group bound every element; products below 2^(-8 S) of (row max * col max) are dropped
    amax = np.abs(a).reshape(3, 2, m, k).max(axis=(1, 3))          # [groups, m]
    bmax = np.abs(b).reshape(3, 2, n, k).max(axis=(1, 3))
    bound = (slices + 2) * 2.0 ** (7 - 8 * slices) * 2 * k * np.einsum("gm,gn->mn", amax, bmax)
    assert (np.abs(c - ref) <= bound + 1e-15 * np.abs(ref).max()).all(), float((np.abs(c - ref) / bound).max())


def test_ozaki_alpha_accumulate_and_zero_rows(torch_cuda):
    rng = np.random.default_rng(11)
    a = rng.standard_normal((3, 140, 40))
    b = rng.standard_normal((3, 70, 40))
    a[:, 5] = 0.0                   # an all-zero row: scale 0
    a[1] = 0.0                      # an all-zero q-slice
    c0 = rng.standard_normal((140, 70))
    c, _ = _ozaki(torch_cuda, a, b, 8, group=1, alpha=-0.5, c0=c0)
    ref = c0 - 0.5 * _ref(a, b)
    assert np.abs(c - ref).max() <= 1e-13 * np.abs(ref).max()
    assert np.array_equal(c[5], c0[5])


def test_ozaki_many_groups_and_splits(torch_cuda):
    """More groups than stages and a split group range (tiles x splits > 148 SMs is not needed for splitting to kick in)."""
    rng = np.random.default_rng(13)
    a = rng.standard_normal((64, 128, 64))
    b = rng.standard_normal((64, 64, 64))
    c, _ = _ozaki(torch_cuda, a, b, 7, group=4)
    ref = _ref(a, b)
    assert np.abs(c - ref).max() <= 1e-12 * np.abs(ref).max()


# ---- the engine's exchange contraction on the emulated path ------------------------------------------------------------
@pytest.mark.parametrize("slices,tol", [(8, 1e-12), (7, 1e-12), (6, 1e-11), (5, 1e-9)])
@pytest.mark.parametrize("method", ["sf", "xtda"])
def test_engine_emulated_exchange(torch_cuda, monkeypatch, slices, tol, method):
    """SF-TDA / X-TDA sigma with the uniform-weight exchange contraction on the INT8 tensor cores against the oracle, with
    several aux chunks (ragged last group: naux = 61), several tiles in M and N, 5 vectors.  The half-transform
    U = Loo . z runs on the INT8 tensor cores too and writes the digit planes of U directly (a-priori row scales)."""
    from oracle import sigma as osig
    from xtddft_b200 import plan as planmod
    from xtddft_b200.engine import SigmaEngine
    from xtddft_b200.synth import make_problem
    monkeypatch.setenv("XTD_CHUNK_AUX", "16")
    p = make_problem(200, 30, 2, 168, 61, 300, xctype="LDA", hyb=0.5, seed=400)
    if method == "sf":
        vind, hd = osig.sf_gen_vind(p, -1, 0)
        plan = planmod.build_sf_plan(p, isf=-1, method=0)
    else:
        vind, hd = osig.xtda_gen_vind(p)
        plan = planmod.build_xtda_plan(p)
    z = np.random.default_rng(1).standard_normal((5, hd.size))
    ref = vind(z)
    eng = SigmaEngine.from_problem(plan, p, workspace_bytes=256 << 20, max_nvec=6, exchange_slices=slices, df_chunk=24)
    got = eng.sigma(torch_cuda.from_numpy(z).cuda()).cpu().numpy()
    assert eng.last_chunks()[0] == 4
    err = float(np.abs(got - ref).max() / max(1.0, np.abs(ref).max()))
    assert err < tol, err
    st = eng.stats()
    assert st["ms"]["k2_slice"] > 0 and st["ms"]["k2"] > 0
    eng.close()


def test_engine_emulated_exchange_ragged_chunks_and_shards(torch_cuda):
    """Chunks that are not multiples of the scale group (the engine carries the remainder over) and a 3-way aux shard whose
    partial buffers must add up to the oracle."""
    import ctypes as C
    from oracle import sigma as osig
    from xtddft_b200 import _lib
    from xtddft_b200 import plan as planmod
    from xtddft_b200.engine import SigmaEngine, _as_tensor
    from xtddft_b200.synth import make_problem
    torch = torch_cuda
    p = make_problem(60, 10, 2, 48, 37, 100, xctype="LDA", hyb=0.5, seed=401)
    vind, hd = osig.sf_gen_vind(p, -1, 0)
    plan = planmod.build_sf_plan(p, isf=-1, method=0)
    z = np.random.default_rng(2).standard_normal((3, hd.size))
    ref = vind(z)
    eng = SigmaEngine.from_problem(plan, p, workspace_bytes=128 << 20, max_nvec=4, exchange_slices=8, df_chunk=13)
    got = eng.sigma_host(z)
    assert np.abs(got - ref).max() < 1e-12 * max(1.0, np.abs(ref).max())
    eng.close()
    zt = torch.from_numpy(z).cuda()
    acc = None
    for r in range(3):
        eng = SigmaEngine.from_problem(plan, p, workspace_bytes=128 << 20, max_nvec=4, rank=r, world=3, exchange_slices=8)
        _lib.check(eng.lib.xtd_sigma_partial(eng._h, 3, C.c_void_p(zt.data_ptr())), "partial")
        ptr, n = C.c_void_p(), C.c_long()
        _lib.check(eng.lib.xtd_partial_buffer(eng._h, 3, C.byref(ptr), C.byref(n)), "buffer")
        part = _as_tensor(torch, ptr.value, n.value, eng.device).clone()
        acc = part if acc is None else acc + part
        if r == 2:
            _as_tensor(torch, ptr.value, n.value, eng.device).copy_(acc)
            out = torch.empty_like(zt)
            _lib.check(eng.lib.xtd_sigma_finish(eng._h, 3, C.c_void_p(out.data_ptr())), "finish")
            assert np.abs(out.cpu().numpy() - ref).max() < 1e-12 * max(1.0, np.abs(ref).max())
        eng.close()


@pytest.mark.parametrize("method,xct", [("sf", "GGA"), ("sf", "LDA"), ("xtda", "LDA"), ("xsf", "GGA")])
def test_engine_emulated_grid_path(torch_cuda, monkeypatch, method, xct):
    """One-component grid kernels (ALDA0 of SF / XSF-TDA, LDA kernels of X-TDA on two channels) with both grid GEMMs on the INT8
    tensor cores: forward Y = phiv . z^T and backward sigma += A^T . phiv (contraction over grid points, several 8192-point
    blocks, ragged last block, two grid chunks) against the oracle."""
    from oracle import sigma as osig
    from xtddft_b200 import plan as planmod
    from xtddft_b200.engine import SigmaEngine
    from xtddft_b200.synth import make_problem
    monkeypatch.setenv("XTD_CHUNK_GRID", "16384")
    p = make_problem(60, 10, 2, 48, 12, 20000, xctype=xct, hyb=0.4, seed=410)
    if method == "sf":
        vind, hd = osig.sf_gen_vind(p, -1, 0)
        plan = planmod.build_sf_plan(p, isf=-1, method=0)
    elif method == "xsf":
        vind, hd = osig.xsf_gen_vind(p, sa=3, method=0, remove=True, foo=0.8, fglobal=0.7)
        plan = planmod.build_sf_plan(p, isf=-1, method=0, sa=3, layout=planmod.LAYOUT_BLOCK, remove=True, foo=0.8, fglobal=0.7, hdiag_kind="xsf")
    else:
        vind, hd = osig.xtda_gen_vind(p)
        plan = planmod.build_xtda_plan(p)
    z = np.random.default_rng(3).standard_normal((3, hd.size))
    ref = vind(z)
    eng = SigmaEngine.from_problem(plan, p, workspace_bytes=512 << 20, max_nvec=4, exchange_slices=7)
    got = eng.sigma(torch_cuda.from_numpy(z).cuda()).cpu().numpy()
    st = eng.stats()
    assert st["ms"]["xc_slice"] > 0, st["ms"]
    assert eng.last_chunks()[1] == 2
    err = float(np.abs(got - ref).max() / max(1.0, np.abs(ref).max()))
    assert err < 1e-11, err
    eng.close()


@pytest.mark.parametrize("nc,no,nv", [(140, 3, 150), (40, 4, 90), (20, 2, 200)])
@pytest.mark.parametrize("sa,remove", [(3, True), (2, False), (1, True)])
def test_engine_emulated_block_weighted_exchange(torch_cuda, monkeypatch, nc, no, nv, sa, remove):
    """XSF-TDA Delta A (block-weighted exchange images): the narrow open-shell output columns keep their DMMA pass, the wide
    virtual block is emulated -- one fused half-transform per occupied row block (closed rows spanning two 128-row tiles, the
    open rows inside a tile), one contraction against the planes of Lvv[v2off:, :].  Several aux chunks, odd / even open-shell
    counts, removed OO vector."""
    from oracle import sigma as osig
    from xtddft_b200 import plan as planmod
    from xtddft_b200.engine import SigmaEngine
    from xtddft_b200.synth import make_problem
    monkeypatch.setenv("XTD_CHUNK_AUX", "8")
    p = make_problem(nc + no + nv, nc, no, nv, 19, 200, xctype="LDA", hyb=0.3, seed=420 + no)
    vind, hd = osig.xsf_gen_vind(p, sa=sa, method=0, remove=remove, foo=0.8, fglobal=0.7)
    plan = planmod.build_sf_plan(p, isf=-1, method=0, sa=sa, layout=planmod.LAYOUT_BLOCK, remove=remove, foo=0.8, fglobal=0.7, hdiag_kind="xsf")
    z = np.random.default_rng(7).standard_normal((3, hd.size))
    ref = vind(z)
    eng = SigmaEngine.from_problem(plan, p, workspace_bytes=512 << 20, max_nvec=4, exchange_slices=7, df_chunk=12)
    got = eng.sigma(torch_cuda.from_numpy(z).cuda()).cpu().numpy()
    assert eng.last_chunks()[0] == 3
    st = eng.stats()
    assert st["ms"]["k2_slice"] > 0, "the emulated path was not taken"
    err = float(np.abs(got - ref).max() / max(1.0, np.abs(ref).max()))
    assert err < 1e-11, err
    assert np.abs(eng.hdiag() - hd).max() < 1e-10
    eng.close()


@pytest.mark.parametrize("method", ["xtda", "sf_mcol"])
@pytest.mark.parametrize("restricted", [True, False])
@pytest.mark.parametrize("short_k", ["0", "512"])
def test_engine_emulated_split_gradient_grid_path(torch_cuda, monkeypatch, method, restricted, short_k):
    """Value + gradient kernels (UKS GGA of X-TDA on two channels, multicollinear GGA spin flip) in the split-gradient form with
    its four value GEMMs on the INT8 tensor cores (two of them batched over the trial vectors), two grid chunks with a ragged
    last block; the streaming kernel between them is the fp64 one.  short_k = 512 (above the occupied count, as the default of 100 is
    here): the occupied-side forward GEMM, whose contraction length is the occupied count, stays on the DMMA GEMM; short_k = 0 forces
    all four onto the INT8 kernel."""
    monkeypatch.setenv("XTD_OZ_SHORT_K", short_k)
    from oracle import sigma as osig
    from xtddft_b200 import plan as planmod
    from xtddft_b200.engine import SigmaEngine
    from xtddft_b200.synth import make_problem
    monkeypatch.setenv("XTD_CHUNK_GRID", "16384")
    p = make_problem(60, 10, 2, 48, 12, 20000, xctype="GGA", hyb=0.4, restricted=restricted, seed=430)
    if method == "xtda":
        vind, hd = osig.xtda_gen_vind(p)
        plan = planmod.build_xtda_plan(p)
    else:
        vind, hd = osig.sf_gen_vind(p, -1, 1)
        plan = planmod.build_sf_plan(p, isf=-1, method=1)
    z = np.random.default_rng(4).standard_normal((3, hd.size))
    ref = vind(z)
    eng = SigmaEngine.from_problem(plan, p, workspace_bytes=1 << 30, max_nvec=4, exchange_slices=7)
    got = eng.sigma(torch_cuda.from_numpy(z).cuda()).cpu().numpy()
    st = eng.stats()
    assert st["ms"]["xc_slice"] > 0, "the emulated grid path was not taken"
    assert eng.last_chunks()[1] == 2
    err = float(np.abs(got - ref).max() / max(1.0, np.abs(ref).max()))
    assert err < 1e-11, err
    eng.close()
