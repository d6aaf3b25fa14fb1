#!/usr/bin/env python3
"""Run a few 2^16 Pallas MSMs (for ncu launch lists): python tools/one_msm.py <window_bits> <chunk>"""
import os, sys
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import srs_fixture
import proof_systems_b200 as zk
from oracle import oracle as orc
wb, chunk = int(sys.argv[1]), int(sys.argv[2])
z = srs_fixture.load("pallas")
g = orc.decompress(orc.PALLAS, z["g_cmp"].tobytes())
sc = orc.random_scalars(orc.FQ, 1 << 16, seed=1)
ctx = zk.Context(0)
ctx.set_option("msm_chunk", chunk)
bases = ctx.upload_bases(zk.PALLAS, g, window_bits=wb)
d = torch.from_numpy(sc.view(np.int64)).cuda()
torch.cuda.synchronize()
for _ in range(4):
    r = ctx.msm_dev(bases, d.data_ptr(), 1 << 16)
print(zk.jacobian_to_affine(zk.PALLAS, r)[:2])
