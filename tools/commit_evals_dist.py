#!/usr/bin/env python3
"""The reference's `IPA Commit Evaluations` bench grid (poly-commitment/benches/ipa.rs:56-130) on the device:
|SRS| = 2^15 (Vesta), evaluations with sparsity {5, 20, 50, 99} % and bit-length {16, 32, 64, 128, 256};
  "com w/o Lagrange" = commit_non_hiding(interpolate(evals), 1)   -> iNTT (host buffer) + MSM on g
  "com Lagrange"     = commit_evaluations_non_hiding(domain, evals) -> MSM on the resident Lagrange basis
Host-side wall time of the public call (pinned-free numpy inputs, result on the host), median of 7; every result is checked
against the oracle.  Writes gpurun_out/commit_evals_dist.json."""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import srs_fixture
import proof_systems_b200 as zk
from oracle import oracle as orc

LOG_N = 15
n = 1 << LOG_N
ctx = zk.Context(0)
z = srs_fixture.load("vesta")
g = ctx.decompress_points(zk.VESTA, z["g_cmp"][:n]) if z["g_cmp"].shape[0] >= n else orc.extend_bases(orc.VESTA, ctx.decompress_points(zk.VESTA, z["g_cmp"]), n)
h = orc.to_mont(orc.FQ, np.ascontiguousarray(z["h_xy"]).view("<u8").reshape(2, 4)).reshape(8)
srs = zk.SRS(ctx, zk.VESTA, g, h)
t0 = time.perf_counter()
lag = srs.get_lagrange_basis_from_domain_size(n)
t_lag = time.perf_counter() - t0
dom = zk.Radix2EvaluationDomain(ctx, zk.FP, n)
rng = np.random.default_rng(5)
m = orc.FP_MODULUS


def med(fn, reps=7):
    ts = []
    for _ in range(reps + 1):
        t = time.perf_counter()
        r = fn()
        ts.append(time.perf_counter() - t)
    return float(np.median(ts[1:])) * 1e3, r


rows = []
for sparsity in (0.05, 0.2, 0.5, 0.99):
    for bitlen in (16, 32, 64, 128, 256):
        vals = orc.limbs_to_ints(orc.random_scalars(orc.FP, n, seed=int(rng.integers(1 << 30))))
        keep = rng.random(n) < sparsity
        ev = [(v % (1 << bitlen)) if k else 0 for v, k in zip(vals, keep)]
        ev_m = orc.to_mont(orc.FP, orc.ints_to_limbs(ev))
        t_a, ca = med(lambda: srs.commit_non_hiding(dom.ifft(ev_m), 1))
        t_b, cb = med(lambda: srs.commit_evaluations_non_hiding(n, ev_m))
        want = orc.msm(orc.VESTA, lag, orc.ints_to_limbs(ev), threads=orc.host_threads())
        ok = bool(np.array_equal(ca.chunks[0], want) and np.array_equal(cb.chunks[0], want))
        rows.append({"sparsity_pct": int(sparsity * 100), "bitlen": bitlen, "interpolate_commit_ms": t_a, "commit_evaluations_ms": t_b, "bit_exact": ok})
        print(rows[-1], flush=True)
rep = {"log_n": LOG_N, "curve": "vesta", "lagrange_basis_build_s": t_lag, "rows": rows}
os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
json.dump(rep, open(os.path.join(ROOT, "gpurun_out", "commit_evals_dist.json"), "w"), indent=1)
assert all(r["bit_exact"] for r in rows)
