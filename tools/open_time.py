#!/usr/bin/env python3
"""Time of SRS::open through zk_srs_open at |g| = 2^16 (Vesta): 45 polynomials in page-locked host memory, the same 45 resident on
the device, and a single polynomial (the rounds alone); stand-in transcript (callbacks return fixed-derivation challenges)."""
import json, os, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import srs_fixture
import proof_systems_b200 as zk
from bench import splitmix64_limbs
LOG_N = int(os.environ.get("LOG_N", "16")); N = 1 << LOG_N
ctx = zk.Context(0)
z = srs_fixture.load("vesta")
g = ctx.decompress_points(zk.VESTA, z["g_cmp"][:N])
srs = zk.SRS(ctx, zk.VESTA, g, g[3])
polys = splitmix64_limbs(5, 45 * N).reshape(45, N, 4)
pin = torch.from_numpy(polys.view(np.int64)).pin_memory()
dev = torch.from_numpy(polys.view(np.int64)).cuda()
bl = splitmix64_limbs(6, 45).reshape(45, 4)
elm, ps, es = splitmix64_limbs(7, 2), splitmix64_limbs(8, 1)[0], splitmix64_limbs(9, 1)[0]
draws = splitmix64_limbs(10, 2 * LOG_N + 2)
chal = splitmix64_limbs(11, LOG_N + 1)
u_base = lambda cip: g[7]
rc = lambda i, l, r: chal[i]
fc = lambda d: chal[-1]
pv = pin.numpy().view(np.uint64)
def run(plnms, reps=5):
    ts = []
    for _ in range(reps + 1):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        zk.srs_open(srs, plnms, elm, ps, es, draws, u_base, rc, fc)
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts[1:])) * 1e3
rows = {}
rows["45 polynomials, page-locked host"] = run([(pv[k], 0, bl[k:k + 1]) for k in range(45)])
rows["45 polynomials, device resident"] = run([((dev.data_ptr() + k * N * 32, N), 0, bl[k:k + 1]) for k in range(45)])
rows["1 polynomial, device resident (the rounds)"] = run([((dev.data_ptr(), N), 0, bl[:1])])
l0 = ctx.launch_count
zk.srs_open(srs, [((dev.data_ptr(), N), 0, bl[:1])], elm, ps, es, draws, u_base, rc, fc)
rows["kernel launches per open"] = ctx.launch_count - l0
print(json.dumps(rows, indent=1))
json.dump(rows, open(os.path.join(ROOT, "gpurun_out", "open_time.json"), "w"), indent=1)
