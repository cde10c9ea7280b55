#!/usr/bin/env python
"""bench.py -- Davidson sigma-vector throughput of the B200-native path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            (N=1 directly; N>1 under torchrun, one rank per GPU)
    python bench.py --impl reference ...                     CPU arm: the oracle port of the reference path on host cores

A "step" is one `vind` call: sigma = A.X for `nvec` trial vectors (default: the workload's number of roots) of
the named BASELINE configuration, on seeded synthetic inputs generated on the device.  At N>1 the auxiliary
functions and grid points are sharded over ranks (strong scaling of the same problem) and every call ends in one
NCCL all-reduce of the MO-space partial sigma.

One JSON line on stdout (rank 0).  `value` = sigma-vectors/s with vectors resident in HBM; `e2e` = the same
through the reference-facing `vind` with HOST vectors (H2D + D2H inside the timed region).  `--steps` / `--warmup` set the
timed and untimed calls of every timed loop (headline, e2e, configs table).

    python bench.py ... --dump-outputs DIR                   also write the last timed step's sigma vectors to DIR/sigma.npy
                                                             (git ignores bench_outputs/)

The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FP64_PEAK_TFLOPS = 37.1      # measured DMMA.8x8x4 issue rate on this pool's B200 (profiles/fp64_peaks_r01.json)


def _hbm_peak():
    """Measured HBM copy bandwidth of this pool's B200s (driver-written MEASURED_PEAKS.json), else the profiling recipe's
    fallback figure."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (torch copy, read+write bytes)"
    except Exception:
        return 6438.8, "fallback: B200 copy bandwidth recorded in BASELINE.md (MEASURED_PEAKS.json absent)"


HBM_PEAK_GBS, HBM_PEAK_SOURCE = _hbm_peak()


def _int8_peak():
    """Dense INT8 tensor-core peak for the emulated exchange contraction.  MEASURED_PEAKS.json holds a measured bf16 figure only;
    the sm_100a tensor core issues int8 (kind::i8, K = 32 per instruction) at twice the bf16 rate (K = 16), so the roofline
    denominator is 2 x the measured SUSTAINED bf16 figure (the kernel runs inside a long, power-capped step)."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        return 2.0 * float(d["bf16_tflops_sustained"]), "2 x MEASURED_PEAKS.json bf16_tflops_sustained (int8 issues at twice the bf16 rate; no measured int8 entry)"
    except Exception:
        return 2.0 * 1400.0, "fallback: 2 x 1.4 PFLOP/s sustained bf16 of the profiling recipe (MEASURED_PEAKS.json absent)"


INT8_PEAK_TOPS, INT8_PEAK_SOURCE = _int8_peak()


def _ncu_traffic(workload: str, key: str, field: str = "traffic_bytes_per_launch"):
    """DRAM bytes per launch of the named kernel from the committed `ncu --set full` capture of this workload
    (profiles/ncu_traffic_r01.json), or None when no capture of this workload exists."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic_r01.json")) as f:
            v = json.load(f)[workload][key][field]
            return float(v) if field == "traffic_bytes_per_launch" else v
    except Exception:
        return None


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=int(os.environ.get("XTD_BENCH_CONFIG", "5")))
    ap.add_argument("--scale", type=float, default=float(os.environ.get("XTD_BENCH_SCALE", "1.0")))
    ap.add_argument("--nvec", type=int, default=0)
    ap.add_argument("--workspace-gb", type=float, default=0.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--davidson", type=int, default=int(os.environ.get("XTD_BENCH_DAVIDSON", "1")))
    ap.add_argument("--configs-table", type=int, default=int(os.environ.get("XTD_BENCH_TABLE", "1")),
                    help="at N=1 with the headline config: append compact records of BASELINE configs 1-4 measured in the same run")
    ap.add_argument("--exchange-slices", type=int, default=int(os.environ.get("XTD_OZAKI", "-1")),
                    help="exchange contraction: 0 = FP64 DMMA, 3..8 = INT8 tensor-core emulation with that many 7-bit digits, -1 = default")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the sigma vectors of the last timed step to DIR/sigma.npy (float64, "
                         f"a fixed seeded sample of columns when larger than {DUMP_LIMIT_BYTES // 10**6} MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the B200 arm computed")
    return args


DUMP_LIMIT_BYTES = 64 * 10**6      # everything --dump-outputs writes, headers included
DUMP_SEED = 20240917


def sample_columns(a: np.ndarray, max_bytes: int, seed: int = DUMP_SEED):
    """`a` itself if it fits in `max_bytes`, else all its rows at a seeded, sorted sample of columns that does.
    Returns (array, column indices or None)."""
    if a.nbytes <= max_bytes:
        return a, None
    ncol = max(1, max_bytes // (a.shape[0] * a.itemsize))
    cols = np.sort(np.random.default_rng(seed).choice(a.shape[1], size=ncol, replace=False))
    return np.ascontiguousarray(a[:, cols]), cols


def dump_outputs(out_dir: str, name: str, a: np.ndarray) -> dict:
    """Write `a` (float64, [rows, cols]) as out_dir/<name>.npy, sampled by columns to stay within DUMP_LIMIT_BYTES."""
    os.makedirs(out_dir, exist_ok=True)
    kept, cols = sample_columns(np.asarray(a, dtype=np.float64), DUMP_LIMIT_BYTES - 4096)
    path = os.path.join(out_dir, f"{name}.npy")
    np.save(path, kept)
    return {"file": path, "shape": list(kept.shape), "full_shape": list(a.shape), "dtype": "float64",
            "columns": "all" if cols is None else f"{cols.size} sampled with numpy default_rng({DUMP_SEED}), sorted"}


# ---------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        # the busy samples: SM clock above the idle floor
        busy = [s for s in sm if s > 500] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------
# CPU arm (oracle port of the reference algorithm), bounded sample + linear extrapolation
# ---------------------------------------------------------------------------------------------------------
def _host_threads():
    """Give the host BLAS every core of the box, whatever the launcher exported (torchrun sets OMP_NUM_THREADS=1, which would
    make the CPU arm an 1-core run): returns (threads in force, BLAS name)."""
    ncpu = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=ncpu)
        info = threadpool_info()
        threads = max([i.get("num_threads", 1) for i in info] or [1])
        blas = ",".join(sorted({i.get("internal_api", "?") for i in info}))
        return int(threads), blas
    except Exception:
        return ncpu, "?"


def cpu_reference_rate(dp, nvec_sample: int = 1, target_s: float = 20.0):
    """Time the oracle's AO-route sigma build (reference algorithm: back-transform, (L_P D) L_P exchange, grid contraction,
    projection) ONCE on all host cores.  If one full-size sigma vector fits the time budget it is timed at full size
    (`extrapolated: false`); otherwise a SAMPLE of the aux functions / grid points sized for the budget is timed and the
    full-size time follows from linearity: t_df * naux / naux_s + t_grid * ng / ng_s + t_rest (`extrapolated: true`)."""
    from oracle import jk, numint
    from xtddft_b200.synth_device import host_sample
    from oracle.workloads import oracle_vind_for
    threads, blas = _host_threads()
    n = dp.p.nao
    # calibrate: host DGEMM rate -> seconds per aux function (~4 N^3 flops per density) and per grid point
    a = np.random.default_rng(0).standard_normal((min(n, 1500), min(n, 1500)))
    _ = a @ a
    t0 = time.perf_counter()
    _ = a @ a
    gf = 2.0 * a.shape[0] ** 3 / (time.perf_counter() - t0) / 1e9
    per_aux = 4.0 * n ** 3 / 1e9 / max(gf, 1.0)
    ndens = 2 if dp.method == "xtda" else (5 if dp.method == "xsf" else 1)
    naux_s = int(max(1, min(dp.naux, (target_s * 0.6) / max(per_aux * ndens, 1e-9))))
    per_g = 4.0 * n ** 2 * (2 if dp.nvar == 4 else 1) / 1e9 / max(gf, 1.0)
    ng_s = int(max(64, min(dp.ng, (target_s * 0.3) / max(per_g * (2 if dp.method == "xtda" else 1), 1e-9))))
    # the sample itself must stay cheap to generate and to hold on the host (seeded NumPy arrays): <= 8 GiB of tensor, <= 4 GiB of AO values
    naux_s = int(min(naux_s, max(1, (8 << 30) // (8 * n * n))))
    ng_s = int(min(ng_s, max(64, (4 << 30) // (8 * n * max(dp.nvar, 1)))))
    full = naux_s == dp.naux and ng_s == dp.ng
    ps = host_sample(dp, naux_s, ng_s)
    vind, hd = oracle_vind_for(ps, dp.method)
    z = np.random.default_rng(1).standard_normal((nvec_sample, hd.size))
    # whole sampled call
    t0 = time.perf_counter(); vind(z); t_all = time.perf_counter() - t0
    if full:
        t_full = t_all / nvec_sample
        return {"value": 1.0 / t_full, "unit": "sigma-vectors/s", "cores": int(threads), "kind": "port", "extrapolated": False,
                "sample": f"oracle AO-route sigma build of {nvec_sample} FULL-SIZE vector(s) ({dp.naux} aux functions, {dp.ng} grid points), "
                          f"timed once; {blas} {threads} threads, host DGEMM {gf:.0f} GF/s",
                "seconds_per_vector_full_size": t_full, "seconds_measured": t_all}
    # parts: exchange/Coulomb on the sampled tensor, grid on the sampled points
    ps_nodf = host_sample(dp, naux_s, ng_s); ps_nodf.cderi = None
    v2, _ = oracle_vind_for(ps_nodf, dp.method) if dp.method != "xsf" else (None, None)
    if v2 is not None:
        t0 = time.perf_counter(); v2(z); t_nodf = time.perf_counter() - t0
        t_df = max(t_all - t_nodf, 1e-9)
    else:
        # XSF needs the tensor for Delta A: time its J/K builds directly (5 densities per vector)
        dm = np.random.default_rng(2).standard_normal((5 * nvec_sample, n, n))
        t0 = time.perf_counter(); jk.get_jk(ps.cderi, dm); t_df = time.perf_counter() - t0
        t_nodf = max(t_all - t_df, 1e-9)
    t_grid = 0.0
    if dp.fxc_kind != "none":
        dm = np.random.default_rng(3).standard_normal((nvec_sample, n, n))
        t0 = time.perf_counter()
        if dp.fxc_kind == "alda0":
            numint.nr_uks_fxc_sf(ps.ao, ps.fxc_alda0, dm)
        elif dp.fxc_kind == "mcol":
            numint.nr_uks_fxc_sf_mc(ps.ao, ps.weights, ps.fxc_mcol, dm)
        else:
            numint.nr_uks_fxc(ps.ao, ps.weights, ps.fxc_uks, np.stack([dm, dm]))
        t_grid = time.perf_counter() - t0
    t_rest = max(t_nodf - t_grid, 0.0)
    t_full = (t_df * dp.naux / naux_s + t_grid * dp.ng / ng_s + t_rest) / nvec_sample
    return {"value": 1.0 / t_full, "unit": "sigma-vectors/s", "cores": int(threads), "kind": "port", "extrapolated": True,
            "sample": f"oracle AO-route sigma build of {nvec_sample} vector(s) on {naux_s}/{dp.naux} aux functions "
                      f"({100.0 * naux_s / dp.naux:.1f} %) and {ng_s}/{dp.ng} grid points ({100.0 * ng_s / dp.ng:.1f} %), timed once and "
                      f"extrapolated linearly (sigma is linear in both); {blas} {threads} threads, host DGEMM {gf:.0f} GF/s; "
                      f"t_df={t_df:.2f}s t_grid={t_grid:.2f}s t_rest={t_rest:.2f}s",
            "seconds_per_vector_full_size": t_full, "seconds_measured": t_all}


def config_dict(dp, nvec: int, dim: int, world: int) -> dict:
    p = dp.p
    return {"workload": dp.name, "method": dp.method, "nvec_per_step": nvec, "nao": p.nao, "nc": p.nc, "no": p.no, "nv": p.nv,
            "dim": dim, "naux": dp.naux, "ng": dp.ng, "grid_components": dp.nvar, "hyb": p.hyb,
            "generator": p.meta.get("generator", "synthetic"),
            "parallelism": f"aux+grid sharded x{world}, one all-reduce of [nvec,dim] per call",
            "l2": "inputs larger than L2 (DF tensor and AO values stream from HBM every call)"}


def run_reference(args):
    """`--impl reference`: the reference's CPU implementation of the path.  PySCF is not installable here (no wheel,
    no network) and the reference tree does not import without it (`baseline/_ref` and `import pyscf` are probed and
    reported), so this arm times the oracle port (kind "port") on ALL host cores -- the BLAS thread count is set explicitly,
    whatever OMP_NUM_THREADS the launcher exported.  One measurement with a ~30 s budget of CPU work (and a sample that
    stays below 12 GiB of host memory): a full-size sigma vector when it fits (configs 1, 2), else a sample of the aux
    functions / grid points extrapolated linearly (`extrapolated: true`);
    `--steps` / `--warmup` do not repeat a minute-long CPU run."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from xtddft_b200.synth_device import make_device_problem
    from xtddft_b200.workloads import plan_for
    dp = make_device_problem(args.config, args.scale)
    nvec = args.nvec or dp.nroots
    cb = cpu_reference_rate(dp, 1, target_s=float(os.environ.get("XTD_REF_BUDGET_S", "30")))
    v = float(cb["value"])
    have_pyscf = False
    try:
        import pyscf  # noqa: F401
        have_pyscf = True
    except Exception:
        pass
    cb["pyscf_importable"] = have_pyscf
    cb["baseline_ref_present"] = os.path.isdir(os.path.join(ROOT, "baseline", "_ref"))
    out = {"impl": "reference", "metric": "davidson_sigma_vectors_per_s", "value": v, "unit": "sigma-vectors/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * nvec / v, "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": "f64", "data": "synthetic", "extrapolated": bool(cb.get("extrapolated")),
           "seconds_measured": cb.get("seconds_measured"),
           "config": config_dict(dp, nvec, int(plan_for(dp.p, dp.method).ext_dim), 1),
           "cpu_baseline": cb, "e2e": {"value": v, "unit": "sigma-vectors/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


def compact_config_record(cfg: int, steps: int = 2, warmup: int = 3, cpu_budget_s: float = 5.0) -> dict:
    """One BASELINE configuration measured like the headline one, reduced to a few numbers: ms per step, sigma-vectors/s, Davidson
    time-to-roots, the dominant phase with its share of the step and its rate, and the CPU baseline (bounded sample)."""
    import torch
    from xtddft_b200.davidson import davidson_for_engine
    from xtddft_b200.synth_device import make_device_problem
    from xtddft_b200.workloads import default_workspace_bytes, engine_for_device_problem
    dp = make_device_problem(cfg, 1.0)
    nvec = dp.nroots
    eng = engine_for_device_problem(dp, max_nvec=max(nvec, 16), workspace_bytes=default_workspace_bytes(dp, 1))
    try:
        dev = eng.device
        g = torch.Generator(device=dev); g.manual_seed(4242)
        z = torch.randn((nvec, eng.ext_dim), generator=g, device=dev, dtype=torch.float64)
        z /= z.norm(dim=1, keepdim=True)
        out = torch.empty_like(z)
        for _ in range(warmup):
            eng.sigma(z, out)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        phase, pflops = {}, {}
        e0.record()
        for _ in range(steps):
            eng.sigma(z, out)
        e1.record()
        torch.cuda.synchronize()
        ms_step = e0.elapsed_time(e1) / steps
        # per-phase times need the eager path (a replayed CUDA graph times only the total): one more call with stats
        eng.sigma(z, out)
        st = eng.stats()
        phase = {k: v for k, v in st["ms"].items() if k != "total" and v > 0}
        pflops = st["flops"]
        rec = {"config": cfg, "workload": dp.name, "method": dp.method, "nvec_per_step": nvec, "dim": int(eng.ext_dim),
               "ms_per_step": ms_step, "sigma_vectors_per_s": nvec / (ms_step * 1e-3), "exchange_slices": int(eng.exchange_slices)}
        if phase:
            top = max(phase, key=phase.get)
            rec["dominant_phase"] = top
            rec["dominant_phase_share"] = phase[top] / max(sum(phase.values()), 1e-12)
            if pflops.get(top, 0.0) > 0:
                rec["dominant_phase_fp64_equiv_tflops"] = pflops[top] / (phase[top] * 1e-3) / 1e12
        warm = eng.ext_dim < 50000
        if warm:          # small problems: one untimed solve first (module loading, graph capture of every call shape)
            davidson_for_engine(eng, dp.nroots, dp.method)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        conv, e, x, info = davidson_for_engine(eng, dp.nroots, dp.method)
        torch.cuda.synchronize()
        rec["davidson"] = {"time_to_roots_s": time.perf_counter() - t0, "nroots": dp.nroots, "converged": bool(np.all(conv)), "warm": warm,
                           "cycles": int(info[0]), "sigma_vectors": int(info[1]), "lowest_root_ha": float(e[0])}
    finally:
        eng.close()
        del eng
        torch.cuda.empty_cache()
    cb = cpu_reference_rate(dp, 1, target_s=cpu_budget_s)
    rec["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "extrapolated", "sample")}
    rec["cpu_baseline"]["time_to_roots_s_extrapolated"] = rec["davidson"]["sigma_vectors"] / cb["value"]
    return rec


def zvector_record(cfg: int = 4, steps: int = 3, warmup: int = 3) -> dict:
    """SURVEY 8f row f3 measured on a BASELINE X-TDA workload's inputs: the Z-vector operator (grad_hb/tdroks_sfu.py:284-321) as one
    engine call per Krylov vector, and a full device solve for a seeded right-hand side."""
    import dataclasses
    import torch
    from xtddft_b200.synth_device import make_device_problem
    from xtddft_b200.workloads import default_workspace_bytes, engine_for_device_problem
    from xtddft_b200.zvector import solve_linear
    dp = dataclasses.replace(make_device_problem(cfg, 1.0), method="zvector")
    eng = engine_for_device_problem(dp, max_nvec=4, workspace_bytes=default_workspace_bytes(dp, 1))
    try:
        dev = eng.device
        g = torch.Generator(device=dev); g.manual_seed(777)
        z = torch.randn((1, eng.ext_dim), generator=g, device=dev, dtype=torch.float64)
        z /= z.norm()
        out = torch.empty_like(z)
        for _ in range(warmup):
            eng.sigma(z, out)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            eng.sigma(z, out)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        st = eng.stats()
        phase = {k: v for k, v in st["ms"].items() if k != "total" and v > 0}
        rhs = torch.randn(eng.ext_dim, generator=g, device=dev, dtype=torch.float64)
        rhs = (rhs / rhs.norm()).cpu().numpy()
        t0 = time.perf_counter()
        x, conv, cycles, res = solve_linear(eng.sigma, rhs, eng.plan.hdiag, tol=1e-8, max_cycle=40)
        torch.cuda.synchronize()
        return {"config": cfg, "workload": dp.name + " inputs, Z-vector equation (row f3)", "method": eng.plan.method, "dim": int(eng.ext_dim),
                "ms_per_operator_call": ms, "phase_ms": phase, "exchange_slices": int(eng.exchange_slices),
                "solve": {"seconds": time.perf_counter() - t0, "cycles": int(cycles), "converged": bool(conv), "residual": float(res),
                          "tol": 1e-8, "rhs": "seeded unit vector"}}
    finally:
        eng.close()
        del eng
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------------------
_JSON_FD = None


def _claim_stdout():
    """Keep stdout for the ONE JSON line: everything else any library prints on fd 1 (e.g. NCCL's version banner) is
    sent to stderr for the rest of the run."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    sys.stdout.flush()
    os.write(_JSON_FD if _JSON_FD is not None else 1, line)


def main():
    args = parse()
    _claim_stdout()
    if args.impl == "reference":
        return run_reference(args)
    import torch
    from xtddft_b200 import _lib
    from xtddft_b200.dist import SigmaReducer, init_process_group_from_env
    from xtddft_b200.synth_device import make_device_problem
    from xtddft_b200.workloads import default_workspace_bytes, engine_for_device_problem

    rank, local_rank, world = init_process_group_from_env()
    if not torch.cuda.is_available():
        raise _lib.XtdError("bench.py needs a B200: the sigma path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    reducer = SigmaReducer() if world > 1 else None
    dp = make_device_problem(args.config, args.scale)
    nvec = args.nvec or dp.nroots
    ws = int(args.workspace_gb * (1 << 30)) if args.workspace_gb > 0 else default_workspace_bytes(dp, world)
    t_setup0 = time.perf_counter()
    xs = None if args.exchange_slices < 0 else args.exchange_slices
    eng = engine_for_device_problem(dp, max_nvec=max(nvec, 16), workspace_bytes=ws, rank=rank, world=world, reducer=reducer,
                                    exchange_slices=xs)
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t_setup0
    dim = eng.ext_dim

    g = torch.Generator(device=dev); g.manual_seed(4242)
    z = torch.randn((nvec, dim), generator=g, device=dev, dtype=torch.float64)
    z /= z.norm(dim=1, keepdim=True)
    out = torch.empty_like(z)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        eng.sigma(z, out)
    barrier()
    eng.stats()                                # drop the all-reduce events of the warm-up calls from the per-phase accounting
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # ---- resident-vector timing -------------------------------------------------------------------------
    eng.reset_stats()
    launches0 = eng.lib.xtd_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    phase, phase_flops = {}, {}
    barrier()
    e0.record()
    for _ in range(args.steps):
        eng.sigma(z, out)
        st = eng.stats()                       # syncs the stream; per-phase device times of this call
        for k, v in st["ms"].items():
            phase[k] = phase.get(k, 0.0) + v
        for k, v in st["flops"].items():
            phase_flops[k] = phase_flops.get(k, 0.0) + v
    e1.record()
    barrier()
    dumped = None
    if args.dump_outputs and rank == 0:
        # what the caller of the timed path receives from the last timed step (all ranks hold the reduced sigma)
        dumped = {"sigma": dump_outputs(args.dump_outputs, "sigma", out.cpu().numpy())}
    ms_total = e0.elapsed_time(e1)
    launches = eng.lib.xtd_launch_count() - launches0
    flops = eng.stats()["flops_gemm"]
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = nvec / (ms_step / 1000.0)
    # ---- end to end: host vectors through the vind boundary ------------------------------------------------
    z_host = z.cpu().numpy()
    if world == 1:
        eng.sigma_host(z_host)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            hz_host = eng.sigma_host(z_host)
        e2e_s = (time.perf_counter() - t0) / args.steps
    else:
        pin_in = torch.from_numpy(z_host).pin_memory()
        pin_out = torch.empty_like(pin_in).pin_memory()
        barrier()
        e0.record()
        for _ in range(args.steps):
            zd = pin_in.to(dev, non_blocking=True)
            pin_out.copy_(eng.sigma(zd), non_blocking=True)
            torch.cuda.synchronize()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        e2e_s = float(t.item()) / 1000.0 / args.steps
    clocks = sampler.stop() if rank == 0 else {}

    # ---- Davidson time-to-roots ---------------------------------------------------------------------------
    dav = None
    if args.davidson:
        try:
            from xtddft_b200.davidson import davidson_for_engine
            warm = dim < 50000
            if warm:      # small problems: the first solve pays one-off costs (CUDA module loading, graph capture of every call shape)
                davidson_for_engine(eng, dp.nroots, dp.method)
            barrier()
            t0 = time.perf_counter()
            tm = {}
            conv, e, x, info = davidson_for_engine(eng, dp.nroots, dp.method, timing=None if warm else tm)
            torch.cuda.synchronize()
            dav = {"time_to_roots_s": time.perf_counter() - t0, "nroots": dp.nroots, "converged": bool(np.all(conv)),
                   "cycles": int(info[0]), "sigma_vectors": int(info[1]), "lowest_root_ha": float(e[0]),
                   "seconds_in_sigma": tm.get("sigma_s"), "warm": warm, "tolerances": "reference SF_TDA.py:392-395 / XTDA.py:775-777 / XSF_TDA.py:1467-1470"}
        except ImportError:
            dav = None

    if rank != 0:
        if world > 1:
            torch.distributed.destroy_process_group()
        return
    # ---- roofline of the dominant kernel (the DMMA GEMM; K2 = exchange contraction launches) -------------------
    # flops the DMMA GEMM executed inside the K2 phase (counted by the engine per launch: 2 M N K nouter batches; equal to
    # 2 naux_loc nvec no nv^2 per exchange term for the uniform-weight methods)
    gemm_ms = phase.get("k2", 0.0) / args.steps
    k2_flops = phase_flops.get("k2", 0.0) / args.steps
    p = dp.p
    xs_on = int(getattr(eng, "exchange_slices", 0) or 0)
    if xs_on and gemm_ms > 0:
        # emulated path: `achieved` counts the int8 multiply-adds the tensor core executes, S(S+1)/2 plane products per fp64 product
        pairs = xs_on * (xs_on + 1) // 2
        tops = k2_flops * pairs / (gemm_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": f"oz_gemm_kernel<{xs_on}> (exchange contraction sigma += U . Lvv emulated on tcgen05.mma kind::i8, "
                                             f"{xs_on} balanced radix-256 digit planes per operand, {pairs} int8 plane products per fp64 product)",
                "achieved": tops, "peak": INT8_PEAK_TOPS, "unit": "TOP/s (int8, dense)", "frac": tops / INT8_PEAK_TOPS,
                "traffic": _ncu_traffic(dp.name, "k2_int8") if world == 1 and args.scale == 1.0 else None, "peak_source": INT8_PEAK_SOURCE,
                "fp64_equivalent_tflops": k2_flops / (gemm_ms * 1e-3) / 1e12,
                "fp64_equivalent_vs_dmma_peak": k2_flops / (gemm_ms * 1e-3) / 1e12 / FP64_PEAK_TFLOPS,
                "fp64_dmma_peak_tflops": FP64_PEAK_TFLOPS,
                "flops_per_launch_group": k2_flops, "int8_ops_per_step": k2_flops * pairs, "ms_per_step_in_kernel": gemm_ms,
                "all_gemm_flops_per_step": flops / args.steps, "all_gemm_tflops_over_step": flops / args.steps / (ms_step * 1e-3) / 1e12}
    else:
      roof = {"bound": "tensor", "kernel": "dgemm_dmma_tma_kernel (exchange contraction sigma += U . Lvv)",
            "achieved": (k2_flops / (gemm_ms * 1e-3) / 1e12) if gemm_ms > 0 else None, "peak": FP64_PEAK_TFLOPS, "unit": "TFLOP/s",
            "frac": (k2_flops / (gemm_ms * 1e-3) / 1e12 / FP64_PEAK_TFLOPS) if gemm_ms > 0 else None,
            "traffic": _ncu_traffic(dp.name, "k2") if world == 1 and args.scale == 1.0 else None,
            "peak_source": "measured DMMA.8x8x4 issue rate, profiles/fp64_peaks_r01.json (MEASURED_PEAKS.json has no FP64 entry; "
                           "cuBLAS DGEMM on the same box: 35.4 TFLOP/s)",
            "flops_per_launch_group": k2_flops, "ms_per_step_in_kernel": gemm_ms,
            "all_gemm_flops_per_step": flops / args.steps, "all_gemm_tflops_over_step": flops / args.steps / (ms_step * 1e-3) / 1e12}
    # SURVEY 8(d): the same exchange build counted with the REFERENCE algorithm's flops (tagged DF-K in the AO basis,
    # 4 naux N^2 nocc per vector and spin block) over the time this build spends on it (K1 + K2): throughput-equivalent
    ref_flops = sum(4.0 * (dp.naux // world + (1 if rank < dp.naux % world else 0)) * p.nao ** 2 * eng.plan.channels[kt.ch].no * nvec
                    for kt in eng.plan.k_terms)
    k_ms = (phase.get("k1", 0.0) + phase.get("k2", 0.0) + phase.get("k2_slice", 0.0)) / args.steps
    try:
        roof["launches_per_step"] = int(eng.last_chunks()[0]) * max(1, len(eng.plan.k_terms))   # one launch per aux chunk and exchange term
    except Exception:
        pass
    if roof["traffic"] is not None:
        roof["traffic_scope"] = "per launch (ONE aux chunk), as ncu reports it; flops_per_launch_group and ms_per_step_in_kernel are per STEP"
        # `traffic` is per LAUNCH (one aux chunk) as ncu reports it; the launch it was captured on, for comparison
        roof["traffic_captured_launch"] = _ncu_traffic(dp.name, "k2_int8" if xs_on else "k2", "captured_launch")
    roof["reference_algorithm_flops_per_step"] = ref_flops
    roof["reference_algorithm_tflops_equivalent"] = (ref_flops / (k_ms * 1e-3) / 1e12) if k_ms > 0 else None
    # ---- streaming kernel of the grid path (xc_weight_kernel) against HBM bandwidth --------------------------
    roof_xc = None
    xs_ms = phase.get("xc_stream", 0.0) / args.steps
    if dp.fxc_kind != "none" and xs_ms > 0:
        ng_loc = dp.ng // world + (1 if rank < dp.ng % world else 0)
        nve = 1 if dp.fxc_kind == "alda0" else dp.nvar
        n_fxc = {"alda0": 1, "mcol": dp.nvar ** 2, "uks": (2 * dp.nvar) ** 2}[dp.fxc_kind]
        occ_cols = sum(ch.no for ch in eng.plan.channels)
        split_form = bool(_lib.check(eng.lib.xtd_xc_split_form(eng._h, nvec), "xtd_xc_split_form"))
        if split_form:
            # per grid point: Y0 read + A written (nvec x no), T read + B written (nvec x nv), 4 occupied and 3 virtual
            # gradient components of the MO values read once, kernel row read once
            vir_cols = sum(ch.nv for ch in eng.plan.channels)
            xc_bytes = 8.0 * ng_loc * (2 * nvec * (occ_cols + vir_cols) + 4 * occ_cols + 3 * vir_cols + n_fxc)
            xc_kernel = "xc_weight_split_kernel (split-gradient form: CTA per grid point, warp per trial vector, MO values staged in smem)"
        else:
            # per grid point: Y read + A written in place (nve components x nvec x no), phi read once, kernel row read once
            xc_bytes = 8.0 * ng_loc * (2 * nve * nvec * occ_cols + nve * occ_cols + n_fxc)
            xc_kernel = "xc_weight_kernel (rho1 on the grid, f_xc weighting, A buffers in place)"
        hbm_peak = HBM_PEAK_GBS
        roof_xc = {"bound": "hbm", "kernel": xc_kernel,
                   "achieved": xc_bytes / (xs_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                   "frac": xc_bytes / (xs_ms * 1e-3) / 1e9 / hbm_peak,
                   "traffic": _ncu_traffic(dp.name, "xc_stream") if world == 1 and args.scale == 1.0 else None, "bytes_per_step": xc_bytes,
                   "ms_per_step_in_kernel": xs_ms, "peak_source": HBM_PEAK_SOURCE}
    out_json = {
        "metric": "davidson_sigma_vectors_per_s", "value": value, "unit": "sigma-vectors/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": dict(config_dict(dp, nvec, dim, world),
                       contraction_arithmetic=(f"fp64 in / fp64 out; dense contractions emulated on the INT8 tensor cores: {xs_on} balanced radix-256 digit "
                                               "planes per operand, exact int32 accumulation, fp64 recombination (sigma equal to the FP64 DMMA path to "
                                               "~4e-16 relative at this size)") if xs_on else "fp64 (DMMA tensor-core GEMM)"),
        "clocks": clocks,
        "e2e": {"value": nvec / e2e_s, "unit": "sigma-vectors/s", "h2d_bytes_per_step": nvec * dim * 8, "d2h_bytes_per_step": nvec * dim * 8},
        "gpu_launches": int(launches),
        "roofline": roof,
        "roofline_xc": roof_xc,
        "phase_ms_per_step": {k: v / args.steps for k, v in phase.items()},
        "setup_s": setup_s,
    }
    if dav is not None:
        out_json["davidson"] = dav
    if dumped is not None:
        out_json["dumped_outputs"] = dumped
    if world == 1 and not args.no_cpu_baseline:
        cb = cpu_reference_rate(dp)
        if dav is not None and cb.get("value"):
            # BASELINE.md section 3: the CPU time-to-roots is EXTRAPOLATED from the CPU rate and the sigma-vector count of the
            # solve above (the CPU never runs the full solve)
            cb["time_to_roots_s_extrapolated"] = dav["sigma_vectors"] / cb["value"]
        out_json["cpu_baseline"] = cb
    if world == 1 and args.configs_table and args.config == 5 and args.scale == 1.0:
        # BASELINE configs 1-4 in the same driver-run record (the headline config needs the whole GPU: release it first)
        eng.close()
        del eng, z, out
        torch.cuda.empty_cache()
        table = []
        for c in (1, 2, 3, 4):
            try:
                table.append(compact_config_record(c, steps=args.steps, warmup=args.warmup))
            except Exception as ex:      # a failed side measurement must not lose the headline record
                table.append({"config": c, "error": f"{type(ex).__name__}: {ex}"})
        try:
            table.append(zvector_record(4, steps=args.steps, warmup=args.warmup))
        except Exception as ex:
            table.append({"config": 4, "method": "zvector_roks", "error": f"{type(ex).__name__}: {ex}"})
        out_json["configs"] = table
    emit(out_json)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
