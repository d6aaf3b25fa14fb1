#!/usr/bin/env python3
"""Device-resident timing sweep (CUDA events around the C-ABI call, L2 flushed between reps):
   MSM: n in {2^11, 2^16, 2^20(Vesta, synthetic extension)} x window bits;   NTT: log_n in 10..20, forward, batch 1 and 16.
Prints a table and writes gpurun_out/sweep.json.  Used to pick defaults and for BASELINE.md's measured tables."""
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import srs_fixture
import proof_systems_b200 as zk
from oracle import oracle as orc

ctx = zk.Context(0)
stream = torch.cuda.Stream()
ctx.set_stream(stream.cuda_stream)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
out = {"msm": [], "ntt": []}


def timed(fn, reps=5):
    ts = []
    for _ in range(reps + 2):
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts[2:]))


which = sys.argv[1] if len(sys.argv) > 1 else "all"
if which in ("all", "msm"):
    z = srs_fixture.load("pallas")
    g = orc.decompress(orc.PALLAS, z["g_cmp"].tobytes())
    chunks = [int(x) for x in os.environ.get("CHUNKS", "16").split(",")]
    for log_n, windows in ((11, (0, 8, 10)), (16, (0, 12, 13, 14, 15, 16))):
        n = 1 << log_n
        sc = orc.random_scalars(orc.FQ, n, seed=1)
        d_sc = torch.from_numpy(sc.view(np.int64)).cuda()
        want = orc.msm(orc.PALLAS, g[:n], sc)
        for wb, chunk in [(w, k) for w in windows for k in chunks]:
            ctx.set_option("msm_chunk", chunk)
            t0 = time.time()
            bases = ctx.upload_bases(zk.PALLAS, g[:n], window_bits=wb)
            up = time.time() - t0
            res = ctx.msm_dev(bases, d_sc.data_ptr(), n)
            ok = bool(np.array_equal(zk.jacobian_to_affine(zk.PALLAS, res), want))
            ms = timed(lambda: ctx.msm_dev(bases, d_sc.data_ptr(), n))
            ctx.set_profile(True)
            ctx.msm_dev(bases, d_sc.data_ptr(), n)
            st = ctx.last_stage_ms()
            ctx.set_profile(False)
            row = {"log_n": log_n, "window_bits": wb, "chunk": chunk, "ms": ms, "points_per_s": n / ms * 1e3, "ok": ok, "upload_s": up,
                   "stages": {k: round(v, 4) for k, v in st.items() if k != "ntt"}}
            out["msm"].append(row)
            print(json.dumps(row), flush=True)
            bases.free()
if which in ("all", "ntt"):
    for log_n in (10, 12, 14, 16, 18, 19, 20):
        n = 1 << log_n
        for batch in (1, 16) if log_n <= 19 else (1,):
            a = torch.from_numpy(orc.to_mont(orc.FP, orc.random_scalars(orc.FP, n * batch, seed=2)).view(np.int64)).cuda()
            ms = timed(lambda: ctx.ntt_dev(zk.FP, a.data_ptr(), log_n, batch=batch))
            row = {"log_n": log_n, "batch": batch, "ms": ms, "elements_per_s": n * batch / ms * 1e3, "GBps_64B_per_elem": 64 * n * batch / ms / 1e6}
            out["ntt"].append(row)
            print(json.dumps(row), flush=True)
os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
json.dump(out, open(os.path.join(ROOT, "gpurun_out", f"sweep_{which}.json"), "w"), indent=1)
