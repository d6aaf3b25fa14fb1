#!/usr/bin/env python3
"""2^16-point Pallas MSM, device-resident scalars: time per MSM and per stage for table windows 14..16 and task-count targets
(msm_wave_threads = accumulation threads per SM the task count is sized for), single MSMs and fused batches of 2 / 7 / 15."""
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
LOG_N = int(os.environ.get("LOG_N", "16")); n = 1 << LOG_N
def timed(fn, reps=9):
    ts = []
    for _ in range(reps + 2):
        flush.fill_(1); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); fn(); e1.record(stream); e1.synchronize(); ts.append(e0.elapsed_time(e1))
    return float(np.median(ts[2:]))
rows = []
sc = splitmix64_limbs(1, 16 * n).reshape(16, n, 4)
d = torch.from_numpy(sc.view(np.int64)).cuda()
for wb in [int(x) for x in os.environ.get("WINDOWS", "14,15,16").split(",")]:
    bases = ctx.upload_bases(zk.PALLAS, g[:n], window_bits=wb)
    for wave in [int(x) for x in os.environ.get("WAVES", "192,256,384,512,768,1024").split(",")]:
        ctx.set_option("msm_wave_threads", wave)
        t = timed(lambda: ctx.msm_dev(bases, d.data_ptr(), n))
        ctx.set_profile(True); ctx.msm_dev(bases, d.data_ptr(), n); st = ctx.last_stage_ms(); ctx.set_profile(False)
        rows.append({"window": wb, "wave_threads": wave, "batch": 1, "ms_per_msm": round(t, 4), "stages_us": {a: round(1e3 * b, 1) for a, b in st.items() if a != "ntt"}})
        print(rows[-1], flush=True)
    ctx.set_option("msm_wave_threads", 0)
    for chunk in [int(x) for x in os.environ.get("CHUNKS", "").split(",") if x]:
        ctx.set_option("msm_chunk", chunk)
        t = timed(lambda: ctx.msm_dev(bases, d.data_ptr(), n))
        ctx.set_profile(True); ctx.msm_dev(bases, d.data_ptr(), n); st = ctx.last_stage_ms(); ctx.set_profile(False)
        rows.append({"window": wb, "chunk": chunk, "batch": 1, "ms_per_msm": round(t, 4), "stages_us": {a: round(1e3 * b, 1) for a, b in st.items() if a != "ntt"}})
        print(rows[-1], flush=True)
    ctx.set_option("msm_chunk", 0)
    for k in [int(x) for x in os.environ.get("BATCHES", "2,7,15").split(",") if x]:
        import ctypes
        from proof_systems_b200._lib import check, _u64p
        out = np.empty((k, 12), dtype=np.uint64)
        h = torch.from_numpy(sc[:k].view(np.int64)).pin_memory()
        t = timed(lambda: check(zk.lib().zk_msm_batch(ctx._h, bases._h, 0, n, ctypes.c_void_p(h.data_ptr()), k, 0, 0, out.ctypes.data_as(_u64p))), reps=5)
        rows.append({"window": wb, "batch": k, "ms_per_msm": round(t / k, 4), "ms_total": round(t, 4), "note": "pinned host scalars through zk_msm_batch"})
        print(rows[-1], flush=True)
    bases.free()
json.dump(rows, open(os.path.join(ROOT, "gpurun_out", "msm_tune.json"), "w"), indent=1)
