#!/usr/bin/env python3
"""The command ncu wraps for profiles/: a few 2^16-point Pallas MSMs (table window from argv[1], default 16), a few 2^20 and 2^16
Fp NTTs, device-resident inputs, nothing else on the GPU."""
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import srs_fixture
import proof_systems_b200 as zk
from bench import splitmix64_limbs
tma_ab = len(sys.argv) > 1 and sys.argv[1] == "msm_tma"      # alternate the two accumulate kernels (profiles/r02_tma_ab.md)
if tma_ab: sys.argv[1] = "16"
wb = int(sys.argv[1]) if len(sys.argv) > 1 else 16
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
ctx = zk.Context(0)
z = srs_fixture.load("pallas")
g = ctx.decompress_points(zk.PALLAS, z["g_cmp"])
bases = ctx.upload_bases(zk.PALLAS, g, window_bits=wb)
d = torch.from_numpy(splitmix64_limbs(1, 1 << 16).view(np.int64)).cuda()
p20 = torch.from_numpy(splitmix64_limbs(2, 1 << 20).view(np.int64)).cuda()
p16 = torch.from_numpy(splitmix64_limbs(2, 1 << 16).view(np.int64)).cuda()
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
for it in range(2 * reps if tma_ab else reps):
    if tma_ab: ctx.set_option("msm_tma", it & 1)
    flush.fill_(1); torch.cuda.synchronize()
    ctx.msm_dev(bases, d.data_ptr(), 1 << 16)
    flush.fill_(1); torch.cuda.synchronize()
    ctx.ntt_dev(zk.FP, p20.data_ptr(), 20)
    ctx.ntt_dev(zk.FP, p16.data_ptr(), 16)
print("done", ctx.launch_count)
