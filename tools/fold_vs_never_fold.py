#!/usr/bin/env python3
"""Direct base fold against never-folded bases, round by round (|g| = 2^16, Vesta), measured on the same machine:
  direct   round j = fold of h = n/2^(j+1) pairs (zk_points_fold_dev, 128-bit challenge = the endo form's length; 255-bit beside it)
           + the L/R pair as two MSMs over h plain points each (no table can exist for bases that change every round)
  never    round j = the L/R pair as one fused batch of two MSMs over the resident window table of the ORIGINAL bases with the
           expanded scalars a[.] * s_j[.] (half of them zero), whatever j
and the 16 rounds of zk_ipa_* for tables of several window widths (the never-fold rounds as shipped)."""
import json, os, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import srs_fixture
import proof_systems_b200 as zk
from bench import splitmix64_limbs
LOG_N = 16; N = 1 << LOG_N
ctx = zk.Context(0)
stream = torch.cuda.Stream(); ctx.set_stream(stream.cuda_stream)
z = srs_fixture.load("vesta")
g = ctx.decompress_points(zk.VESTA, z["g_cmp"][:N])
def timed(fn, reps=7):
    ts = []
    for _ in range(reps + 2):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); fn(); e1.record(stream); e1.synchronize(); ts.append(e0.elapsed_time(e1))
    return float(np.median(ts[2:]))
out = {"direct": [], "never_fold_rounds_by_table_window": {}}
d_g, d_out = ctx.dev_alloc(N * 64), ctx.dev_alloc(N * 32)
ctx.dev_upload(d_g, g)
u128 = np.array([0x9e3779b97f4a7c15, 0xbf58476d1ce4e5b9, 0, 0], dtype=np.uint64)
u255 = splitmix64_limbs(3, 1)[0]; u255[3] &= (1 << 61) - 1
sc = torch.from_numpy(splitmix64_limbs(5, 2 * N).reshape(2, N, 4).view(np.int64)).cuda()
for j in range(LOG_N):
    h = N >> (j + 1)
    t128 = timed(lambda: ctx.points_fold_dev(zk.VESTA, d_g, h, u128, d_out))
    t255 = timed(lambda: ctx.points_fold_dev(zk.VESTA, d_g, h, u255, d_out))
    plain = ctx.upload_bases(zk.VESTA, g[:max(h, 1)], window_bits=0)
    tm = timed(lambda: (ctx.msm_dev(plain, sc[0].data_ptr(), h), ctx.msm_dev(plain, sc[1].data_ptr(), h)))
    plain.free()
    out["direct"].append({"round": j, "h": h, "fold_128bit_ms": round(t128, 4), "fold_255bit_ms": round(t255, 4), "lr_two_plain_msms_ms": round(tm, 4)})
    print(out["direct"][-1], flush=True)
ctx.dev_free(d_g); ctx.dev_free(d_out)
a, b, us = splitmix64_limbs(1, N), splitmix64_limbs(2, N), splitmix64_limbs(3, 2 * LOG_N)
for wb in (12, 13, 14, 15, 16):
    bases = ctx.upload_bases(zk.VESTA, g, window_bits=wb)
    ts = []
    for rep in range(4):
        r = zk.IpaRounds(ctx, bases, a, b)
        torch.cuda.synchronize(); t0 = time.perf_counter()
        for j in range(LOG_N):
            r.lr(); r.fold(us[2 * j], us[2 * j + 1])
        torch.cuda.synchronize(); ts.append(1e3 * (time.perf_counter() - t0))
        r.close()
    out["never_fold_rounds_by_table_window"][wb] = round(float(np.median(ts[1:])), 3)
    print("never-fold, table window", wb, "16 rounds ms", out["never_fold_rounds_by_table_window"][wb], flush=True)
    bases.free()
tot128 = sum(r["fold_128bit_ms"] + r["lr_two_plain_msms_ms"] for r in out["direct"])
out["direct_total_ms_128bit"] = round(tot128, 3)
print("direct fold, 16 rounds (128-bit challenges):", out["direct_total_ms_128bit"], "ms")
json.dump(out, open(os.path.join(ROOT, "gpurun_out", "fold_vs_never_fold.json"), "w"), indent=1)
