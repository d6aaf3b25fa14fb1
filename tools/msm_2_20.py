#!/usr/bin/env python3
"""BASELINE config 4 timing: 2^20-point Vesta MSM (fixture generators extended deterministically), resident window-16 table,
uniform Fp scalars seed 3; device-resident scalars, CUDA events, L2 flushed.  Also the per-shard time of an 8-way split."""
import json, os, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import srs_fixture
import proof_systems_b200 as zk
from oracle import oracle as orc
ctx = zk.Context(0)
stream = torch.cuda.Stream(); ctx.set_stream(stream.cuda_stream)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
z = srs_fixture.load("vesta")
n = 1 << 20
g = orc.extend_bases(orc.VESTA, ctx.decompress_points(zk.VESTA, z["g_cmp"]), n)
sc = orc.random_scalars(orc.FP, n, seed=3)
t0 = time.time(); bases = ctx.upload_bases(zk.VESTA, g, window_bits=-1); up = time.time() - t0
d = torch.from_numpy(sc.view(np.int64)).cuda()
def timed(fn, reps=5):
    ts = []
    for _ in range(reps + 2):
        flush.fill_(1); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); fn(); e1.record(stream); e1.synchronize(); ts.append(e0.elapsed_time(e1))
    return float(np.median(ts[2:]))
full = timed(lambda: ctx.msm_dev(bases, d.data_ptr(), n))
ctx.set_profile(True); ctx.msm_dev(bases, d.data_ptr(), n); st = ctx.last_stage_ms(); ctx.set_profile(False)
shard = timed(lambda: ctx.msm_dev(bases, d.data_ptr(), n // 8, off=0))
t0 = time.time(); want = orc.msm(orc.VESTA, g, sc, threads=orc.host_threads()); cpu = time.time() - t0
ok = bool(np.array_equal(zk.jacobian_to_affine(zk.VESTA, ctx.msm_dev(bases, d.data_ptr(), n)), want))
rep = {"n": n, "window_bits": bases.window_bits, "table_upload_s": up, "ms": full, "points_per_s": n / full * 1e3, "stages_ms": st,
       "shard_1_of_8_ms": shard, "cpu_oracle_s": cpu, "cpu_threads": orc.host_threads(), "bit_exact": ok}
print(json.dumps(rep))
json.dump(rep, open(os.path.join(ROOT, "gpurun_out", "msm_2_20.json"), "w"), indent=1)
