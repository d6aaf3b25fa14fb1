#!/usr/bin/env python3
"""Diagnostic for the weak-scaling step at N ranks (torchrun): per rank and per step, the device time of (a) the plain resident MSM,
(b) the sharded MSM with the library's exchange, ranks aligned before every step; SM clocks of every rank's GPU during the loop."""
import json, os, sys, threading, time
import numpy as np, torch, torch.distributed as dist
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import srs_fixture
import proof_systems_b200 as zk
from proof_systems_b200.parallel import LibraryComm
from bench import splitmix64_limbs
rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
ctx = zk.Context(local)
stream = torch.cuda.Stream(); ctx.set_stream(stream.cuda_stream)
z = srs_fixture.load("pallas")
g = ctx.decompress_points(zk.PALLAS, z["g_cmp"])
n = 1 << 16
bases = ctx.upload_bases(zk.PALLAS, g, window_bits=16)
d = torch.from_numpy(splitmix64_limbs(rank + 1, n).view(np.int64)).cuda()
comm = LibraryComm(ctx)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
clocks = []
stop = False
def poll():
    import pynvml
    pynvml.nvmlInit()
    h = pynvml.nvmlDeviceGetHandleByIndex(local)
    while not stop:
        clocks.append(int(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))); time.sleep(0.02)
th = threading.Thread(target=poll, daemon=True); th.start()
def run(fn, steps, align):
    ts = []
    for _ in range(steps):
        flush.fill_(rank + 1); torch.cuda.synchronize()
        if align:
            dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); fn(); e1.record(stream); e1.synchronize(); ts.append(round(e0.elapsed_time(e1), 3))
    return ts
for _ in range(5):
    comm.msm(bases, d.data_ptr(), n); ctx.msm_dev(bases, d.data_ptr(), n)
res = {"rank": rank}
res["plain"] = run(lambda: ctx.msm_dev(bases, d.data_ptr(), n), 12, False)
res["sharded_aligned"] = run(lambda: comm.msm(bases, d.data_ptr(), n), 12, True)
res["sharded_unaligned"] = run(lambda: comm.msm(bases, d.data_ptr(), n), 12, False)
# the exchange alone: a 2 KB all-gather through torch's communicator, aligned
buf_in = torch.zeros(256, dtype=torch.int64, device="cuda"); buf_out = torch.zeros(256 * world, dtype=torch.int64, device="cuda")
def ag():
    with torch.cuda.stream(stream):
        dist.all_gather_into_tensor(buf_out, buf_in)
res["torch_allgather_2KB_aligned"] = run(ag, 12, True)
stop = True; th.join(timeout=1)
res["sm_mhz_min_med_max"] = [min(clocks), sorted(clocks)[len(clocks) // 2], max(clocks)] if clocks else None
out = [None] * world
dist.all_gather_object(out, res)
if rank == 0:
    for r in out: print(json.dumps(r))
    json.dump(out, open(os.path.join(ROOT, "gpurun_out", "diag_scale.json"), "w"), indent=1)
dist.destroy_process_group()
