"""Z-vector right-hand side and W matrix at full size: config-4 inputs (make_device_problem(4, 1.0), method "zvector") on one GPU.

Records the time of `rhs` + `w_matrix` for one state (CUDA-synchronised wall clock, plus the device phase split of every
`xtd_block_response` call), its ratio to one operator application, the device memory in use (cudaMemGetInfo) before the engine,
after it, and the least free memory seen during rhs / w_matrix, and whether the whole-MO-space route's first engine can be built at
this size.  Writes one JSON file:  python profiles/scripts/zvector_rhs_bench.py OUT.json"""
import dataclasses
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def main(out_path):
    import torch
    from xtddft_b200 import plan as planmod
    from xtddft_b200.engine import SigmaEngine
    from xtddft_b200.synth_device import make_device_problem
    from xtddft_b200.workloads import default_workspace_bytes
    from xtddft_b200.zvector import assemble_rhs, assemble_w, block_callables, rhs_intermediates
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    rec = {"gpu": gpu, "config": 4}
    dp = dataclasses.replace(make_device_problem(4, 1.0), method="zvector")
    p = dp.p
    rec.update(nc=p.nc, no=p.no, nv=p.nv, naux=dp.naux, ng=dp.ng, xctype=p.xctype, hyb=p.hyb)
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
    rec["exchange_slices"] = eng.exchange_slices
    rec["device_bytes_engine"] = free0 - free1
    # one operator application
    z = torch.randn((1, eng.ext_dim), dtype=torch.float64, device=eng.device)
    for _ in range(2):
        eng.sigma(z)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        eng.sigma(z)
    e1.record()
    torch.cuda.synchronize()
    rec["ms_operator"] = e0.elapsed_time(e1) / 3
    calls, low = [], [free1]

    def apply_blocks(d, c, x):
        t0 = time.perf_counter()
        r = eng.block_response(d, c, x)
        torch.cuda.synchronize()
        st = eng.stats()
        low.append(torch.cuda.mem_get_info()[0])
        calls.append({"coef": [float(v) for v in c], "x": x is not None, "seconds": time.perf_counter() - t0, "chunks": eng.last_chunks(),
                      "phase_ms": {k: v for k, v in st["ms"].items() if v > 0}})
        return r
    resp, sfx, full = block_callables(p, plan, apply_blocks)
    rng = np.random.default_rng(4)
    v = rng.standard_normal((p.nc, p.nv))
    v /= np.linalg.norm(v)
    zz = rng.standard_normal(eng.ext_dim)
    for rep in range(2):                    # the first pass warms up; the second is recorded
        calls.clear()
        t0 = time.perf_counter()
        inter = rhs_intermediates(p, v, resp, sfx)
        rhs = assemble_rhs(p, v, None, None, inter=inter)
        t1 = time.perf_counter()
        im0 = assemble_w(p, zz, inter, full)
        t2 = time.perf_counter()
    rec.update(seconds_rhs=t1 - t0, seconds_w=t2 - t1, calls=calls, finite=bool(np.isfinite(rhs).all() and np.isfinite(im0).all()))
    rec["ratio_to_operator"] = (t2 - t0) * 1e3 / rec["ms_operator"]
    rec["device_bytes_in_use_peak"] = free0 - min(low)
    eng.close()
    del eng
    torch.cuda.empty_cache()
    # the whole-MO-space route: its first engine (general J / K / f_xc response on nmo x nmo channels)
    try:
        mp = planmod.build_mo_response_plan(p, range_separated=False)
        free2, _ = torch.cuda.mem_get_info()
        e = SigmaEngine(mp, p.nao, p.mo_coeff, workspace_bytes=1 << 30)
        dp.make_grid(e, 0, 1)
        e.grid_commit()
        dp.stream_cderi(e, 0, 0, 1)
        e.finalize(1)
        torch.cuda.synchronize()
        rec["mo_space"] = {"fits": True, "device_bytes_first_engine": free2 - torch.cuda.mem_get_info()[0]}
        e.close()
    except Exception as ex:                 # an allocation the device cannot satisfy is reported by the engine, not faulted
        rec["mo_space"] = {"fits": False, "error": f"{type(ex).__name__}: {ex}"[:400]}
    with open(out_path, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({k: rec[k] for k in ("ms_operator", "seconds_rhs", "seconds_w", "ratio_to_operator", "device_bytes_engine",
                                          "device_bytes_in_use_peak", "mo_space")}))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "zvector_rhs_cfg4.json")
