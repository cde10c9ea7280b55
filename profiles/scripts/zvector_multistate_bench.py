"""Z-vectors of k states at once against k states one at a time: config-4 inputs (make_device_problem(4, 1.0), method "zvector",
GGA, default emulated exchange) on one GPU.

For k = 1, 2, 4, 8 seeded states it times right-hand side + solve + W matrix
  * "batched": `block_callables_many` / `per_state_batched` (one `xtd_block_response_batch` call per image for all k states) and
    `solve_linear_block` (operator calls of up to max_nvec = 4 vectors);
  * "single": today's calls per state (`block_callables`, `solve_linear`, one vector per operator call),
alternating the two (single first, then batched, twice for k <= 4, once for k = 8).  Recorded per run: CUDA-synchronised wall time,
the device time of the engine calls (sum of the engine's own `total` event pair after every block-response and operator call), the
operator calls, the solver cycles, the largest difference between the two solutions, and the device memory in use (cudaMemGetInfo)
before the engine and at its lowest free point.  GPU name, power limit and SM clock are read at the start and at the end.
Writes one JSON file:  python profiles/scripts/zvector_multistate_bench.py OUT.json"""
import dataclasses
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def _gpu_state():
    q = "name,power.limit,power.draw,clocks.sm,clocks.max.sm,temperature.gpu"
    return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()


def main(out_path):
    import torch
    from xtddft_b200 import plan as planmod
    from xtddft_b200.engine import SigmaEngine
    from xtddft_b200.synth_device import make_device_problem
    from xtddft_b200.workloads import default_workspace_bytes
    from xtddft_b200.zvector import (assemble_rhs, assemble_w, block_callables, block_callables_many, per_state_batched,
                                     rhs_intermediates, solve_linear, solve_linear_block)
    rec = {"gpu_start": _gpu_state(), "config": 4}
    dp = dataclasses.replace(make_device_problem(4, 1.0), method="zvector")
    p = dp.p
    rec.update(nc=p.nc, no=p.no, nv=p.nv, naux=dp.naux, ng=dp.ng, xctype=p.xctype, hyb=p.hyb, restricted=bool(p.restricted))
    torch.cuda.synchronize()
    free0, total = torch.cuda.mem_get_info()
    plan = planmod.build_zvector_plan(p)
    plan.block_response = True
    eng = SigmaEngine(plan, p.nao, p.mo_coeff, workspace_bytes=default_workspace_bytes(dp, 1))
    dp.make_grid(eng, 0, 1)
    eng.grid_commit()
    torch.cuda.empty_cache()
    dp.stream_cderi(eng, 0, 0, 1)
    eng.finalize(4)
    torch.cuda.synchronize()
    free1, _ = torch.cuda.mem_get_info()
    rec.update(exchange_slices=eng.exchange_slices, dim=eng.ext_dim, device_bytes_in_use_before_engine=total - free0,
               device_bytes_in_use_with_engine=total - free1)
    hdiag = np.asarray(plan.hdiag)
    tol, max_cycle = (1e-12 if p.restricted else 1e-8), 40
    sign = 1.0 if p.restricted else -1.0
    acc = {"device_ms": 0.0, "low": free1}

    def counted(fn):
        def f(*a, **kw):
            r = fn(*a, **kw)
            torch.cuda.synchronize()
            acc["device_ms"] += eng.stats()["ms"]["total"]
            acc["low"] = min(acc["low"], torch.cuda.mem_get_info()[0])
            return r
        return f
    block_response, sigma = counted(eng.block_response), counted(eng.sigma)

    def run_single(V, Z):
        rhs, zs, ws, cyc = [], [], [], []
        for v in V:
            resp, sfx, full = block_callables(p, plan, block_response)
            inter = rhs_intermediates(p, v, resp, sfx)
            r = assemble_rhs(p, v, None, None, inter=inter)
            z, conv, c, res = solve_linear(sigma, sign * r, hdiag, tol=tol, max_cycle=max_cycle)
            ws.append(assemble_w(p, z, inter, full))
            rhs.append(r), zs.append(z), cyc.append(int(c))
        return np.stack(zs), {"operator_calls": int(sum(cyc)), "cycles": cyc}

    def run_batched(V, Z):
        k = len(V)
        resp, sfx, full = block_callables_many(p, plan, block_response)
        inters = per_state_batched(k, lambda i, r, x: rhs_intermediates(p, V[i], r, x), resp, sfx)
        rhs = np.stack([assemble_rhs(p, V[i], None, None, inter=it) for i, it in enumerate(inters)])
        z, conv, cyc, res, calls = solve_linear_block(sigma, sign * rhs, hdiag, tol=tol, max_cycle=max_cycle, max_nvec=eng.max_nvec)
        per_state_batched(k, lambda i, f: assemble_w(p, z[i], inters[i], f), full)
        return z, {"operator_calls": int(calls), "cycles": [int(c) for c in cyc], "converged": [bool(c) for c in conv]}

    def timed(fn, V, Z):
        acc["device_ms"], acc["low"] = 0.0, torch.cuda.mem_get_info()[0]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        z, info = fn(V, Z)
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        info.update(seconds=sec, seconds_per_state=sec / len(V), device_ms=acc["device_ms"], device_ms_per_state=acc["device_ms"] / len(V),
                    device_bytes_in_use_peak=total - acc["low"])
        return z, info

    rng = np.random.default_rng(4)
    V8 = rng.standard_normal((8, p.nc, p.nv))
    V8 /= np.linalg.norm(V8, axis=(1, 2), keepdims=True)
    timed(run_single, V8[:1], None)                    # warm-up of every shape: one state each way
    timed(run_batched, V8[:2], None)
    runs = []
    for k in (1, 2, 4, 8):
        for rep in range(2 if k <= 4 else 1):
            zs, si = timed(run_single, V8[:k], None)
            zb, bi = timed(run_batched, V8[:k], None)
            diff = float(np.abs(zb - zs).max() / max(1.0, np.abs(zs).max()))
            runs.append({"k": k, "rep": rep, "single": si, "batched": bi, "max_rel_diff_solutions": diff})
            print(json.dumps({"k": k, "rep": rep, "single_s_per_state": round(si["seconds_per_state"], 3),
                              "batched_s_per_state": round(bi["seconds_per_state"], 3), "calls": [si["operator_calls"], bi["operator_calls"]],
                              "diff": diff}), flush=True)
    rec["runs"] = runs
    rec["gpu_end"] = _gpu_state()
    eng.close()
    with open(out_path, "w") as f:
        json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "zvector_multistate_cfg4.json")
