#!/usr/bin/env python3
"""diagnostic: concurrent host callers on the lane pool vs the oracle"""
import os, sys, threading, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import srs_fixture
import proof_systems_b200 as zk
from oracle import oracle as orc
z = srs_fixture.load("pallas")
n, k = 1 << 14, 15
c = zk.Context(0)
g = c.decompress_points(zk.PALLAS, z["g_cmp"][:n])
bases = c.upload_bases(zk.PALLAS, g, window_bits=-1)
sc = [orc.random_scalars(orc.FQ, n, seed=300 + j) for j in range(k)]
want = [orc.msm(orc.PALLAS, g, sc[j]) for j in range(k)]
aff = lambda r: zk.jacobian_to_affine(zk.PALLAS, r)
for lanes in (4, 1, 2, 4):
    c.set_option("ctx_lanes", lanes)
    ser = [aff(c.msm(bases, sc[j])) for j in range(k)]
    print("lanes", lanes, "serial mismatches vs oracle:", [j for j in range(k) if not np.array_equal(ser[j], want[j])], flush=True)
    for nthreads in (2, 4, 15):
        bad_total = 0
        for rep in range(5):
            out = [None] * k
            def work(j0):
                for j in range(j0, k, nthreads):
                    out[j] = aff(c.msm(bases, sc[j]))
            th = [threading.Thread(target=work, args=(t,)) for t in range(nthreads)]
            t0 = time.perf_counter()
            for t in th: t.start()
            for t in th: t.join()
            dt = time.perf_counter() - t0
            bad = [j for j in range(k) if not np.array_equal(out[j], want[j])]
            bad_total += len(bad)
        print("lanes", lanes, "threads", nthreads, "mismatches over 5 reps:", bad_total, "last", bad, f"{dt*1e3:.2f} ms", flush=True)
