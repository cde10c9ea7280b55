"""Core-valence-separated X-TDA on config-4 inputs (make_device_problem(4, 1.0): 958 basis functions, nc 136, no 1, nv 821, GGA,
default exchange path) on one GPU, next to the valence config-4 step.

Cases, in this order and repeated `--reps` times so that the valence step and the CVS cases alternate:
  * "valence": the full X-TDA plan, one sigma step of the workload's nroots vectors;
  * "cvs<n>" for n = 1, 2, 4: the CVS plan on the n highest closed orbitals; sigma steps of 20 and 60 vectors and Davidson runs
    (`davidson_for_engine`, X-TDA solver settings) for 20 and 60 roots.
Recorded per case: ms per sigma call (CUDA events over `--steps` calls after `--warmup` calls), the per-phase device times of one more
eager call (`SigmaEngine.stats`), seconds to roots and Davidson cycles / sigma vectors, device memory in use (cudaMemGetInfo) before
the engine, with the engine, and at the lowest free point during the case.  GPU name, power limit and SM clock are read at the start
and at the end.  Writes one JSON file:  python profiles/scripts/cvs_xtda_bench.py OUT.json [--reps 2] [--steps 5] [--warmup 2]"""
import argparse
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


def _engine(dp, plan, max_nvec):
    from xtddft_b200.engine import SigmaEngine
    from xtddft_b200.workloads import default_workspace_bytes
    eng = SigmaEngine(plan, dp.p.nao, dp.p.mo_coeff, workspace_bytes=default_workspace_bytes(dp, 1))
    dp.make_grid(eng, 0, 1)
    eng.grid_commit()
    eng.torch.cuda.empty_cache()
    dp.stream_cderi(eng, 0, 0, 1)
    eng.finalize(max_nvec)
    return eng


def _step(torch, eng, nvec, steps, warmup, seed):
    g = torch.Generator(device=eng.device)
    g.manual_seed(seed)
    z = torch.randn((nvec, eng.ext_dim), generator=g, device=eng.device, dtype=torch.float64)
    z /= z.norm(dim=1, keepdim=True)
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
    # one more call on a fresh output buffer (eager, so the engine times every phase) of at most max_nvec vectors: one engine call
    zz = z[:eng.max_nvec].contiguous()
    eng.sigma(zz, torch.empty_like(zz))
    st = eng.stats()
    return {"nvec": nvec, "ms_per_call": ms, "phase_nvec": int(zz.shape[0]), "phase_ms": {k: v for k, v in st["ms"].items() if v > 0},
            "launches": st["launches"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    import torch
    from xtddft_b200 import plan as planmod
    from xtddft_b200.davidson import davidson_for_engine
    from xtddft_b200.synth_device import make_device_problem
    dp = make_device_problem(4, 1.0)
    p = dp.p
    rec = {"gpu_start": _gpu_state(), "config": 4, "nc": p.nc, "no": p.no, "nv": p.nv, "naux": dp.naux, "ng": dp.ng, "xctype": p.xctype,
           "hyb": p.hyb, "restricted": bool(p.restricted), "valence_nroots": dp.nroots, "steps": args.steps, "warmup": args.warmup}
    cases = [("valence", None)] + [(f"cvs{n}", list(range(p.nc - n, p.nc))) for n in (1, 2, 4)]
    runs = []
    for rep in range(args.reps):
        for name, core in cases:
            torch.cuda.empty_cache()
            torch.cuda.synchronize()
            free0, total = torch.cuda.mem_get_info()
            t0 = time.perf_counter()
            plan = planmod.build_xtda_plan(p, core=core)
            eng = _engine(dp, plan, max_nvec=max(dp.nroots, 40) if core is None else 40)
            torch.cuda.synchronize()
            r = {"case": name, "rep": rep, "core": core, "dim": int(eng.ext_dim), "exchange_slices": int(eng.exchange_slices),
                 "engine_setup_s": time.perf_counter() - t0, "device_bytes_in_use_before_engine": total - free0}
            low = free1 = torch.cuda.mem_get_info()[0]
            r["device_bytes_in_use_with_engine"] = total - free1
            try:
                if core is None:
                    r["sigma"] = [_step(torch, eng, dp.nroots, args.steps, args.warmup, 4242)]
                else:
                    r["sigma"] = [_step(torch, eng, n, args.steps, args.warmup, 4242 + n) for n in (20, 60)]
                    r["davidson"] = []
                    for nroots in (20, 60):
                        torch.cuda.synchronize()
                        t1 = time.perf_counter()
                        conv, e, x, info = davidson_for_engine(eng, nroots, "xtda")
                        torch.cuda.synchronize()
                        low = min(low, torch.cuda.mem_get_info()[0])
                        r["davidson"].append({"nroots": nroots, "seconds_to_roots": time.perf_counter() - t1, "cycles": int(info[0]),
                                              "sigma_vectors": int(info[1]), "converged": int(np.sum(conv)), "e_min": float(np.min(e)),
                                              "e_max": float(np.max(e))})
                low = min(low, torch.cuda.mem_get_info()[0])
                r["device_bytes_in_use_peak_sampled"] = total - low
            finally:
                eng.close()
                del eng
            runs.append(r)
            print(json.dumps({"case": name, "rep": rep, "ms": [round(s["ms_per_call"], 2) for s in r["sigma"]],
                              "dav": [(d["nroots"], round(d["seconds_to_roots"], 2), d["cycles"]) for d in r.get("davidson", [])],
                              "GB": round(r["device_bytes_in_use_with_engine"] / 1e9, 2)}), flush=True)
    rec["runs"] = runs
    rec["gpu_end"] = _gpu_state()
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
