#!/usr/bin/env python3
"""A/B of the accumulation kernel's gather: plain per-lane 64-byte loads (k_accumulate) against the bulk asynchronous copy engine
(k_accumulate_tma: cp.async.bulk + mbarrier, two stages per lane).  2^16-point Pallas MSM, device-resident scalars, tables
w = 15 / 16, L2 flushed between iterations; reports the whole MSM and the accumulate stage, and checks the two give the same point."""
import json, os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import srs_fixture
import proof_systems_b200 as zk
from bench import splitmix64_limbs
ctx = zk.Context(0)
stream = torch.cuda.Stream(); ctx.set_stream(stream.cuda_stream)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
z = srs_fixture.load("pallas")
g = ctx.decompress_points(zk.PALLAS, z["g_cmp"])
n = 1 << 16
def timed(fn, reps=15):
    ts = []
    for _ in range(reps + 3):
        flush.fill_(1); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); fn(); e1.record(stream); e1.synchronize(); ts.append(e0.elapsed_time(e1))
    return float(np.median(ts[3:]))
d = torch.from_numpy(splitmix64_limbs(7, n).view(np.int64)).cuda()
rows = []
for wb in (15, 16):
    bases = ctx.upload_bases(zk.PALLAS, g[:n], window_bits=wb)
    pts = {}
    for tma in (0, 1, 0, 1):
        ctx.set_option("msm_tma", tma)
        t = timed(lambda: ctx.msm_dev(bases, d.data_ptr(), n))
        accs = []
        for _ in range(7):
            flush.fill_(1); torch.cuda.synchronize()
            ctx.set_profile(True); pts[tma] = zk.jacobian_to_affine(zk.PALLAS, ctx.msm_dev(bases, d.data_ptr(), n)); accs.append(ctx.last_stage_ms()["accumulate"]); ctx.set_profile(False)
        rows.append({"window": wb, "gather": "tma" if tma else "ldg", "msm_ms": round(t, 4), "accumulate_us": round(1e3 * float(np.median(accs)), 1)})
        print(rows[-1], flush=True)
    rows.append({"window": wb, "same_point": bool(np.array_equal(pts[0], pts[1]))}); print(rows[-1], flush=True)
    ctx.set_option("msm_tma", 0)
    bases.free()
json.dump(rows, open(os.path.join(ROOT, "gpurun_out", "msm_tma_ab.json"), "w"), indent=1)
