#!/usr/bin/env python3
"""Device-resident MSM time and per-stage breakdown for n = 2^8 .. 2^16 (Pallas, default table window), uniform scalars and
kimchi-like witness columns (mostly 1, a few zeros and random values).  Shows the latency floor of the pipeline."""
import json, os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import srs_fixture
import proof_systems_b200 as zk
from bench import splitmix64_limbs
ctx = zk.Context(0)
if os.environ.get("MSM_CHUNK"): ctx.set_option("msm_chunk", int(os.environ["MSM_CHUNK"]))
if os.environ.get("MSM_WAVE"): ctx.set_option("msm_wave_threads", int(os.environ["MSM_WAVE"]))
WINDOW = int(os.environ.get("MSM_WINDOW", "-1"))
KS = [int(x) for x in os.environ.get("MSM_LOGS", "8,10,11,12,13,14,15,16").split(",")]
stream = torch.cuda.Stream(); ctx.set_stream(stream.cuda_stream)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
z = srs_fixture.load("pallas")
g = ctx.decompress_points(zk.PALLAS, z["g_cmp"])
def timed(fn, reps=7):
    ts = []
    for _ in range(reps + 2):
        flush.fill_(1); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); fn(); e1.record(stream); e1.synchronize(); ts.append(e0.elapsed_time(e1))
    return float(np.median(ts[2:]))
rows = []
for k in KS:
    n = 1 << k
    bases = ctx.upload_bases(zk.PALLAS, g[:n], window_bits=WINDOW)
    for kind in ("uniform", "ones"):
        sc = splitmix64_limbs(k, n)
        if kind == "ones":
            sc[: n - 3] = 0; sc[: n - 10, 0] = 1
        d = torch.from_numpy(sc.view(np.int64)).cuda()
        t = timed(lambda: ctx.msm_dev(bases, d.data_ptr(), n))
        ctx.set_profile(True); ctx.msm_dev(bases, d.data_ptr(), n); st = ctx.last_stage_ms(); ctx.set_profile(False)
        rows.append({"log_n": k, "scalars": kind, "window": bases.window_bits, "ms": round(t, 4), "stages_us": {a: round(1e3 * b, 1) for a, b in st.items()}})
        print(rows[-1], flush=True)
    bases.free()
json.dump(rows, open(os.path.join(ROOT, "gpurun_out", os.environ.get("MSM_OUT", "msm_sizes.json")), "w"), indent=1)
