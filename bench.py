#!/usr/bin/env python3
"""bench.py — Pallas MSM points/s (+ Fp NTT elements/s) at 2^16 on B200, next to the CPU oracle on the same host.

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA library through its C ABI)
    python bench.py --impl reference --gpus N ...            # CPU arm: the oracle port of the reference's ark MSM/FFT
    torchrun --nproc-per-node N bench.py --gpus N ...        # N > 1: one rank per GPU

A "step" is one pass of the hot path over one batch of synthetic input: one 2^16-point Pallas MSM (BASELINE config 2)
followed by one 2^16-element Fp NTT.  The headline metric is the MSM's points/s; the NTT is reported in `ntt`.
  value  : inputs already resident in HBM, device time per step from CUDA events on the launching stream
  e2e    : the same step through the host-pointer C-ABI calls (zk_msm / zk_ntt_batch): scalars and polynomial start in
           PINNED host memory, H2D and D2H inside the timed region
N > 1 (weak scaling): every rank holds the SRS and runs its own 2^16-point slice of an (N * 2^16)-point MSM; the N
partials stay on the device as c slice sums (128 B each), are exchanged with one NCCL all_gather enqueued behind the kernels and
summed on the device (proof_systems_b200/parallel.py: ShardedMsm).  NTT: N independent replicas.
Between timed iterations a 256 MiB buffer is overwritten to flush the 126 MB L2.
--dump-outputs DIR writes what the last timed step returned (see dump_outputs), so that two builds can be compared on identical
inputs: every input is derived from fixed seeds and the fixture's SRS.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: nothing is written there

LOG_N = 16
N_PTS = 1 << LOG_N
MSM_BYTES_PER_POINT = 96      # 64 B affine base + 32 B scalar (SURVEY.md §8d)
NTT_BYTES_PER_ELEM = 64       # 32 B read + 32 B write per transform


def load_traffic():
    p = os.path.join(ROOT, "profiles", "traffic.json")
    return json.load(open(p)) if os.path.exists(p) else {}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + clock-event reasons DURING the timed region: one NVML query between every two timed steps, from the main thread,
    outside the CUDA-event span.  (A polling thread — every 2 ms, then every 10 ms — was measured to stall a step by ~3 ms whenever
    a query coincided with it: NVML and the CUDA runtime share driver locks, and on an 8-GPU box with 8 ranks one such stall per
    20-step leg cost 0.17 ms per step on every rank, tools/diag_scale.py.)  nvidia-smi is the fallback when NVML cannot be loaded."""
    NAMES = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")

    def __init__(self, index=0):
        self.index, self.samples, self.h, self.nv = index, [], None, None
        self.sm_max = None
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if visible:
                ids = [x for x in visible.split(",") if x.strip() != ""]
                if index < len(ids) and ids[index].strip().isdigit():
                    phys = int(ids[index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nv = pynvml
            self.sm_max = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None

    def sample(self):
        """one query; called between timed steps (the GPU has just run a step and the L2 flush)"""
        if self.h is None:
            return
        nv = self.nv
        masks = (nv.nvmlClocksEventReasonHwSlowdown, nv.nvmlClocksEventReasonHwThermalSlowdown,
                 nv.nvmlClocksEventReasonSwThermalSlowdown, nv.nvmlClocksEventReasonSwPowerCap)
        try:
            mhz = int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            try:
                r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            self.samples.append((mhz, tuple(bool(r & m) for m in masks)))
        except Exception:
            pass

    def start(self):
        self.samples = []

    def stop(self):
        if self.h is None:
            return self._smi_once()
        sm = sorted(s[0] for s in self.samples)
        reasons = [n for i, n in enumerate(self.NAMES) if any(s[1][i] for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.sm_max, "reasons": reasons, "samples": len(sm),
                "source": "NVML, one query between every two timed steps (outside the event span)"}

    def _smi_once(self):
        """fallback: one nvidia-smi query right after the timed region"""
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        for query in (q, "clocks.sm,clocks.max.sm"):
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={query}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=20).stdout.strip().splitlines()
                parts = [x.strip() for x in out[0].split(",")]
                if parts[0].isdigit():
                    reasons = [n for i, n in enumerate(self.NAMES) if len(parts) > 2 + i and parts[2 + i].lower().startswith("active")]
                    return {"sm_mhz": int(parts[0]), "sm_max_mhz": int(parts[1]), "reasons": reasons, "samples": 1,
                            "source": "nvidia-smi, one query after the timed region (NVML unavailable)"}
            except Exception:
                continue
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}


def splitmix64_limbs(seed, n):
    """n synthetic field elements: 4 splitmix64 words each, top limb masked to 62 bits (uniform below 2^254 < m).
    Used as canonical MSM scalars and, read as Montgomery residues, as NTT input (every value < m is a valid residue)."""
    idx = np.arange(1, 4 * n + 1, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + idx * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    w = z.reshape(n, 4).copy()
    w[:, 3] &= np.uint64((1 << 62) - 1)
    return w


def compressed_srs():
    """the reference's own srs/pallas.srs generators (compressed, 33 B each), rebuilt by tests/golden/srs_fixture.py"""
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import srs_fixture
    return srs_fixture.load("pallas")["g_cmp"]


def make_inputs(decompress, rank):
    """Pallas SRS generators + seeded scalars / polynomial.  `decompress`: the product's device decoder (our arm) or the
    oracle's (reference arm)."""
    g = decompress(compressed_srs())
    scalars = splitmix64_limbs(1 + rank, N_PTS)      # canonical (msm_bigint form)
    poly = splitmix64_limbs(2, N_PTS)                # Montgomery residues
    return g, scalars, poly


def field_digits(limbs: np.ndarray) -> np.ndarray:
    """u64 limbs [..., 4] of 256-bit values -> float32 [..., 16]: 16 little-endian 16-bit digits per value, exact in float32"""
    return np.ascontiguousarray(limbs, dtype=np.uint64).view(np.uint16).astype(np.float32)


def dump_outputs(out_dir, msm_affine, ntt_out):
    """The headline's last timed step, as float32 digits (field_digits) of the library's Montgomery limbs:
      msm.npy  [2, 16]       the 2^16-point Pallas MSM, converted from the returned Jacobian point to affine (x, y) so that
                             equal points compare equal
      ntt.npy  [2^16, 16]    the polynomial the in-place Fp NTT left on the device (the step transforms the previous step's
                             output: after W warm-up and K timed steps it holds NTT^(W+K) of the seeded input)"""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "msm.npy"), field_digits(np.asarray(msm_affine).reshape(2, 4)))
    np.save(os.path.join(out_dir, "ntt.npy"), field_digits(ntt_out))


def cpu_time(fn, min_seconds, max_reps):
    reps, t0 = 0, time.perf_counter()
    while True:
        fn()
        reps += 1
        el = time.perf_counter() - t0
        if el >= min_seconds or reps >= max_reps:
            return el / reps, reps


def cpu_msm(orc, g, scalars, threads):
    """what SRS::commit_non_hiding runs for a |g|-coefficient polynomial: two half MSMs under rayon::join, then add"""
    return orc.msm_split2(orc.PALLAS, g, scalars, threads=threads)


def best_threads(fn, max_threads):
    """The GPU boxes expose 64-128 hardware threads that are not always all usable (shared host, cgroup quota): after one untimed
    warm-up (OpenMP pool start-up, page faults), run the CPU arm twice per candidate thread count and keep the count with the best
    of its two runs — the baseline gets its best configuration, picked from warmed measurements."""
    best, best_t = None, None
    cand = sorted({t for t in (8, 16, 32, 64, 128, max_threads) if t <= max_threads} or {max_threads})
    fn(cand[-1])
    for t in cand:
        el = None
        for _ in range(2):
            t0 = time.perf_counter()
            fn(t)
            d = time.perf_counter() - t0
            el = d if el is None else min(el, d)
        if best is None or el < best:
            best, best_t = el, t
    return best_t


def bench_config(n_gpus: int, window_bits: int) -> dict:
    """The workload both arms run, worded once so that the two JSON lines carry the same `config` (arm-specific settings live under
    `arm`).  `pippenger_window_bits` is BASELINE config 2's w: the GPU arm's table window; the CPU arm's Pippenger picks ark-ec's own."""
    wl = "2^16-point Pallas MSM on srs/pallas.srs generators, uniform Fq scalars (BASELINE config 2)"
    if n_gpus > 1:
        wl += (f"; {n_gpus} ranks, every rank holds the same 2^16 bases and its own 2^16 scalars (the sum over ranks of <s_r, g>): weak scaling, "
               "one all-gather of the ranks' slice sums (GPU arm: ncclAllGather issued by the library; CPU arm: rank 0 computes one rank's share)")
    return {"workload": wl, "pippenger_window_bits": window_bits,
            "l2": "GPU arm: 256 MiB buffer overwritten between timed iterations (flush); CPU arm: n/a"}


def run_reference(args):
    """The reference's CPU path for this workload, as restated by the oracle (oracle/pasta_oracle.c: ark-style signed-digit
    Pippenger with window-parallel threads; ark-style radix-2 FFT), all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    g, scalars, poly = make_inputs(lambda c: orc.decompress(orc.PALLAS, c.tobytes()), 0)
    threads = best_threads(lambda t: cpu_msm(orc, g, scalars, t), orc.host_threads())
    for _ in range(max(1, args.warmup)):
        cpu_msm(orc, g, scalars, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_msm(orc, g, scalars, threads)
    msm_s = (time.perf_counter() - t0) / args.steps
    t0 = time.perf_counter()
    for _ in range(args.steps):
        orc.ntt(orc.FP, poly, threads=threads)
    ntt_s = (time.perf_counter() - t0) / args.steps
    val = N_PTS / msm_s
    sample = f"{args.steps} x (one 2^16-point Pallas MSM, uniform scalars) after {max(1, args.warmup)} warm-up"
    line = {
        "impl": "reference", "metric": "pallas_msm_points_per_s", "value": val, "unit": "points/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": msm_s * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u256 (4 x u64 Montgomery limbs)", "data": "synthetic",
        "config": bench_config(args.gpus, args.window_bits),
        "arm": {"cpu_path": "oracle port of ark-ec 0.5 msm_bigint under the reference's 2-way rayon::join split (ipa.rs:652-662); the reference is Rust and there is no cargo in the image"},
        "cpu_baseline": {"value": val, "unit": "points/s", "cores": threads, "kind": "port", "sample": sample, "host_threads_available": orc.host_threads()},
        "e2e": {"value": val, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "ntt": {"metric": "fp_ntt_elements_per_s", "value": N_PTS / ntt_s, "unit": "elements/s", "ms": ntt_s * 1e3,
                "workload": "2^16-element Fp forward NTT", "cores": threads},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--window-bits", type=int, default=16, help="table window of the resident SRS for the headline (16 = BASELINE config 2's w; -1: library default)")
    ap.add_argument("--cpu-seconds", type=float, default=6.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--no-extra", action="store_true", help="skip the cfg1 / cfg3 / cfg4 legs (tools/ use this for quick A/B runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (CUDA arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA arm")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    import ctypes

    import torch
    import torch.distributed as dist

    import proof_systems_b200 as zk
    from proof_systems_b200._lib import _u64p, check
    from proof_systems_b200.parallel import LibraryComm, shard_bounds

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: proof_systems_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    ctx = zk.Context(local)
    g, scalars, poly = make_inputs(lambda c: ctx.decompress_points(zk.PALLAS, c), rank)   # inputs come from the product itself
    stream = torch.cuda.Stream(device=local)
    ctx.set_stream(stream.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def flush_l2():
        flush.fill_(rank + 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, collective=False):
        """per-step CUDA events on the launching stream, L2 flushed between steps (outside the timed span); total ms.
        collective: the step contains a cross-rank exchange — the ranks are aligned before every step"""
        tot = 0.0
        for _ in range(steps):
            flush_l2()
            if rank == 0:
                sampler.sample()        # the GPU is busy with the flush right behind the previous step: clocks under load
            torch.cuda.synchronize()
            if world > 1 and collective:
                # every rank enters the step together: the untimed flush / host work of the slowest rank must not be billed to the
                # others' collective (at N = 8 that skew was +0.3 ms per step); the rendezvous itself is outside the event span
                dist.barrier()
                torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            tot += e0.elapsed_time(e1)
        return tot

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def upload_timed(curve, pts, wb):
        """resident bases + their window table; returns (bases, milliseconds of zk_bases_upload incl. the table build)"""
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        b = ctx.upload_bases(curve, pts, window_bits=wb)
        torch.cuda.synchronize()
        return b, (time.perf_counter() - t0) * 1e3

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()     # covers every timed region below

    # =============================================================== headline: cfg2, 2^16-point Pallas MSM (+ the 2^16 Fp NTT)
    bases, table_ms = upload_timed(zk.PALLAS, g, args.window_bits)
    wb = bases.window_bits
    d_scalars = torch.from_numpy(scalars.view(np.int64)).cuda()
    d_poly = torch.from_numpy(poly.view(np.int64)).cuda()
    h_scalars = torch.from_numpy(scalars.view(np.int64)).pin_memory()
    h_poly = torch.from_numpy(poly.view(np.int64).copy()).pin_memory()
    # N > 1 (weak scaling): the exchange is the library's own (csrc/comm.cu): zk_msm_sharded leaves the slice sums on the device,
    # enqueues ONE ncclAllGather of N x c x 128 bytes from C on the context's stream behind the kernels, adds the partials on the
    # device and reads them back once.  torch.distributed only carried the 128-byte NCCL id at start-up.
    comm = LibraryComm(ctx) if world > 1 else None

    def msm_host(b, h_sc, n):
        out = np.empty(12, dtype=np.uint64)
        check(zk.lib().zk_msm(ctx._h, b._h, 0, n, ctypes.c_void_p(h_sc.data_ptr()), 0, 0, out.ctypes.data_as(_u64p)))
        return out

    def step_resident():
        if comm:
            return comm.msm(bases, d_scalars.data_ptr(), N_PTS)
        return ctx.msm_dev(bases, d_scalars.data_ptr(), N_PTS)

    def step_e2e():
        if comm:
            return comm.msm(bases, h_scalars.data_ptr(), N_PTS)   # page-locked scalars are read over PCIe by the first kernel
        return msm_host(bases, h_scalars, N_PTS)

    def ntt_resident():
        ctx.ntt_dev(zk.FP, d_poly.data_ptr(), LOG_N)

    def ntt_e2e():
        check(zk.lib().zk_ntt_batch(ctx._h, zk.FP, ctypes.c_void_p(h_poly.data_ptr()), LOG_N, 1, 0, 0, 0))

    result = None
    for _ in range(args.warmup):
        result = step_resident()
        ntt_resident()
        step_e2e()
        ntt_e2e()
    barrier()
    launches0 = ctx.launch_count
    last = {}

    def step_resident_kept():
        last["msm"] = step_resident()

    msm_ms = timed(step_resident_kept, args.steps, collective=True)
    result = last["msm"]
    barrier()
    ntt_ms = timed(ntt_resident, args.steps)
    if args.dump_outputs:
        stream.synchronize()
        last["ntt"] = d_poly.cpu().numpy().view(np.uint64).reshape(N_PTS, 4).copy()
    barrier()
    msm_e2e_ms = timed(step_e2e, args.steps, collective=True)
    barrier()
    ntt_e2e_ms = timed(ntt_e2e, args.steps)
    barrier()
    launches_total = ctx.launch_count - launches0

    def stage_profile(fn_msm, reps):
        """dominant-kernel durations, live, with CUDA events inside the library (profiling mode, separate pass)"""
        ctx.set_profile(True)
        acc, st = [], None
        for _ in range(reps):
            flush_l2()
            torch.cuda.synchronize()
            fn_msm()
            st = ctx.last_stage_ms()
            acc.append(st["accumulate"])
        ctx.set_profile(False)
        return float(np.median(acc)), {k: v for k, v in st.items() if k != "ntt"}

    def ntt_profile(fn, reps):
        ctx.set_profile(True)
        v = []
        for _ in range(reps):
            flush_l2()
            torch.cuda.synchronize()
            fn()
            v.append(ctx.last_stage_ms()["ntt"])
        ctx.set_profile(False)
        return float(np.median(v))

    acc_ms, stages = stage_profile(lambda: ctx.msm_dev(bases, d_scalars.data_ptr(), N_PTS), min(args.steps, 10))
    ntt_k = ntt_profile(ntt_resident, min(args.steps, 10))
    msm_ms, ntt_ms = max_over_ranks(msm_ms), max_over_ranks(ntt_ms)
    msm_e2e_ms, ntt_e2e_ms = max_over_ranks(msm_e2e_ms), max_over_ranks(ntt_e2e_ms)

    peak, peak_src = load_peaks()
    traffic = load_traffic()
    extra = {"table_build_ms": {f"pallas_2^16_w{wb}": round(table_ms, 3)}}
    ok_all = True

    # =============================================================== second figure: the library's own window choice for 2^16
    if not args.no_extra and world == 1:
        b2, t2 = upload_timed(zk.PALLAS, g, -1)
        for _ in range(3):
            r2 = ctx.msm_dev(b2, d_scalars.data_ptr(), N_PTS)
        t_res = timed(lambda: ctx.msm_dev(b2, d_scalars.data_ptr(), N_PTS), args.steps) / args.steps
        t_e2e = timed(lambda: msm_host(b2, h_scalars, N_PTS), args.steps) / args.steps
        a2, st2 = stage_profile(lambda: ctx.msm_dev(b2, d_scalars.data_ptr(), N_PTS), 5)
        same = bool(np.array_equal(zk.jacobian_to_affine(zk.PALLAS, r2), zk.jacobian_to_affine(zk.PALLAS, result)))
        ok_all &= same
        extra["tuned_window"] = {"window_bits": b2.window_bits, "ms_per_step": t_res, "value": N_PTS / (t_res * 1e-3), "e2e_ms_per_step": t_e2e,
                                 "e2e_value": N_PTS / (t_e2e * 1e-3), "stage_ms": st2, "same_point_as_headline": same}
        extra["table_build_ms"][f"pallas_2^16_w{b2.window_bits}"] = round(t2, 3)
        b2.free()
        # ---- cfg1: 2^11 points of the same SRS (latency floor of the pipeline)
        n1 = 1 << 11
        b1 = ctx.upload_bases(zk.PALLAS, g[:n1], window_bits=-1)
        for _ in range(3):
            r1 = ctx.msm_dev(b1, d_scalars.data_ptr(), n1)
        t1 = timed(lambda: ctx.msm_dev(b1, d_scalars.data_ptr(), n1), args.steps) / args.steps
        t1e = timed(lambda: msm_host(b1, h_scalars, n1), args.steps) / args.steps
        _, st1 = stage_profile(lambda: ctx.msm_dev(b1, d_scalars.data_ptr(), n1), 5)
        extra["cfg1_pallas_2^11"] = {"workload": "2^11-point Pallas MSM on srs/pallas.srs generators (BASELINE config 1)", "window_bits": b1.window_bits,
                                     "ms_per_step": t1, "value": n1 / (t1 * 1e-3), "e2e_ms_per_step": t1e, "stage_ms": st1, "_result": r1}
        b1.free()

    # =============================================================== cfg3: 2^20 Fp NTT, forward + inverse round trip
    if not args.no_extra:
        L3 = 20
        n3 = 1 << L3
        p3 = splitmix64_limbs(2, n3)
        d3_0 = torch.from_numpy(p3.view(np.int64)).cuda()
        d3 = d3_0.clone()

        def roundtrip():
            ctx.ntt_dev(zk.FP, d3.data_ptr(), L3)
            ctx.ntt_dev(zk.FP, d3.data_ptr(), L3, inverse=True)
        for _ in range(3):
            roundtrip()
        rt_ms = max_over_ranks(timed(roundtrip, args.steps)) / args.steps
        stream.synchronize()
        rt_exact = bool(torch.equal(d3, d3_0))
        ctx.ntt_dev(zk.FP, d3.data_ptr(), L3)
        stream.synchronize()                      # the library runs on `stream`; torch's copy below does not
        fwd3 = d3.cpu().numpy().view(np.uint64).reshape(n3, 4)
        d3.copy_(d3_0)
        k3 = ntt_profile(lambda: ctx.ntt_dev(zk.FP, d3.data_ptr(), L3), 5)
        ach3 = NTT_BYTES_PER_ELEM * n3 / (k3 * 1e-3) / 1e9
        tr20 = traffic.get("k_ntt_pass_2_20", {})
        extra["cfg3_fp_ntt_2^20"] = {
            "workload": "2^20-element Fp NTT forward + inverse round trip (BASELINE config 3)" + ("" if world == 1 else f", {world} replicas"),
            "ms_per_round_trip": rt_ms, "value": world * 2 * n3 / (rt_ms * 1e-3), "unit": "elements/s (2 transforms per round trip)",
            "round_trip_bit_exact": rt_exact,
            "roofline": {"bound": "hbm", "kernel": "k_ntt_pass x2 (one forward transform)", "achieved": ach3, "peak": peak, "unit": "GB/s", "frac": ach3 / peak,
                         "traffic": (tr20.get("bytes_per_launch", 0) * tr20.get("launches_per_transform", 0)) or None, "kernel_ms": k3,
                         "algorithmic_bytes": NTT_BYTES_PER_ELEM * n3}}
        ok_all &= rt_exact
        del d3, d3_0

    # =============================================================== cfg4: 2^20-point Vesta MSM, STRONG scaling over the ranks
    if not args.no_extra:
        L4 = 20
        n4 = 1 << L4
        lo, hi = shard_bounds(n4, world, rank)
        pts4 = ctx.synthetic_points(zk.VESTA, n4, seed=4)              # every rank derives the same 2^20 points; keeps its slice
        sc4 = splitmix64_limbs(3, n4)
        b4, t4 = upload_timed(zk.VESTA, pts4[lo:hi], 16)
        d_sc4 = torch.from_numpy(sc4[lo:hi].view(np.int64)).cuda()
        h_sc4 = torch.from_numpy(sc4[lo:hi].view(np.int64).copy()).pin_memory()
        sh4 = comm.msm if comm else (lambda bb, ptr, cnt: ctx.msm_dev(bb, ptr, cnt) if ptr == d_sc4.data_ptr() else msm_host(bb, h_sc4, cnt))
        steps4 = args.steps
        for _ in range(3):
            r4 = sh4(b4, d_sc4.data_ptr(), hi - lo)
        barrier()
        t4_res = max_over_ranks(timed(lambda: sh4(b4, d_sc4.data_ptr(), hi - lo), steps4, collective=True)) / steps4
        barrier()
        t4_e2e = max_over_ranks(timed(lambda: sh4(b4, h_sc4.data_ptr(), hi - lo), steps4, collective=True)) / steps4
        barrier()
        a4, st4 = stage_profile(lambda: ctx.msm_dev(b4, d_sc4.data_ptr(), hi - lo), 3)
        ach4 = MSM_BYTES_PER_POINT * (hi - lo) / (a4 * 1e-3) / 1e9
        extra["cfg4_vesta_2^20_strong"] = {
            "workload": f"2^20-point Vesta MSM split by points over {world} GPU(s) (BASELINE config 4; poly-commitment/benches/msm.rs:92-140), "
                        "synthetic on-curve bases, uniform Fp scalars; slice sums exchanged with one ncclAllGather issued by the library (zk_msm_sharded) and summed on the device",
            "scaling": "strong", "window_bits": b4.window_bits, "points_per_rank": hi - lo, "ms_per_step": t4_res, "value": n4 / (t4_res * 1e-3),
            "unit": "points/s", "e2e_ms_per_step": t4_e2e, "e2e_value": n4 / (t4_e2e * 1e-3), "h2d_bytes_per_step_per_rank": (hi - lo) * 32,
            "stage_ms_rank0": st4,
            "roofline": {"bound": "hbm", "kernel": "k_accumulate (rank 0's slice)", "achieved": ach4, "peak": peak, "unit": "GB/s", "frac": ach4 / peak, "traffic": None,
                         "kernel_ms": a4, "algorithmic_bytes": MSM_BYTES_PER_POINT * (hi - lo)}}
        extra["table_build_ms"][f"vesta_2^{(hi - lo).bit_length() - 1}_w{b4.window_bits}"] = round(t4, 3)
    clocks = sampler.stop() if rank == 0 else None
    if comm:
        barrier()
        comm.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- correctness of what was timed + CPU baseline on the same host (bounded sample): the only use of the oracle
    from oracle import oracle as orc
    threads = best_threads(lambda t: cpu_msm(orc, g, scalars, t), orc.host_threads())
    if world == 1:
        want = orc.msm(orc.PALLAS, g, scalars)
    else:
        tot = [0] * N_PTS
        m = orc.FQ_MODULUS
        for r in range(world):
            sr = orc.limbs_to_ints(splitmix64_limbs(1 + r, N_PTS))
            tot = [(a + b) % m for a, b in zip(tot, sr)]
        want = orc.msm(orc.PALLAS, g, orc.ints_to_limbs(tot))
    ok = bool(np.array_equal(zk.jacobian_to_affine(zk.PALLAS, result), want))
    ok_all &= ok
    cpu_msm_s, cpu_reps = cpu_time(lambda: cpu_msm(orc, g, scalars, threads), args.cpu_seconds, 50)
    cpu_ntt_s, cpu_ntt_reps = cpu_time(lambda: orc.ntt(orc.FP, poly, threads=threads), args.cpu_seconds / 3, 200)
    if "cfg1_pallas_2^11" in extra:
        c1 = extra["cfg1_pallas_2^11"]
        t0 = time.perf_counter()
        w1 = orc.msm(orc.PALLAS, g[:1 << 11], scalars[:1 << 11])
        c1["cpu_oracle_ms"] = (time.perf_counter() - t0) * 1e3
        c1["result_matches_cpu_oracle"] = bool(np.array_equal(zk.jacobian_to_affine(zk.PALLAS, c1.pop("_result")), w1))
        ok_all &= c1["result_matches_cpu_oracle"]
    if "cfg3_fp_ntt_2^20" in extra:
        t0 = time.perf_counter()
        w3 = orc.ntt(orc.FP, p3, threads=threads)
        c3 = extra["cfg3_fp_ntt_2^20"]
        c3["cpu_oracle_forward_ms"] = (time.perf_counter() - t0) * 1e3
        c3["forward_matches_cpu_oracle"] = bool(np.array_equal(fwd3, w3))
        ok_all &= c3["forward_matches_cpu_oracle"]
    if "cfg4_vesta_2^20_strong" in extra:
        t0 = time.perf_counter()
        w4 = orc.msm(orc.VESTA, pts4, sc4, threads=threads)
        c4 = extra["cfg4_vesta_2^20_strong"]
        c4["cpu_oracle_ms"] = (time.perf_counter() - t0) * 1e3
        c4["cpu_oracle_threads"] = threads
        c4["result_matches_cpu_oracle"] = bool(np.array_equal(zk.jacobian_to_affine(zk.VESTA, r4), w4))
        ok_all &= c4["result_matches_cpu_oracle"]

    msm_traffic = traffic.get(f"k_accumulate_w{wb}", traffic.get("k_accumulate", {}) if wb == 15 else {}).get("bytes_per_launch")
    ntt_traffic = traffic.get("k_ntt_pass", {})
    ntt_traffic = ntt_traffic.get("bytes_per_launch", 0) * ntt_traffic.get("launches_per_transform", 0) or None
    per_step_ms = msm_ms / args.steps
    value = world * N_PTS / (per_step_ms * 1e-3)
    e2e_value = world * N_PTS / (msm_e2e_ms / args.steps * 1e-3)
    achieved = MSM_BYTES_PER_POINT * N_PTS / (acc_ms * 1e-3) / 1e9
    ntt_ach = NTT_BYTES_PER_ELEM * N_PTS / (ntt_k * 1e-3) / 1e9
    nwin = (256 + wb - 1) // wb if wb else 1
    line = {
        "metric": "pallas_msm_points_per_s", "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": per_step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u256 (8 x u32 Montgomery limbs)", "data": "synthetic",
        "config": bench_config(world, args.window_bits),
        "arm": {"window_bits": wb, "resident_table_mib": round(len(bases) * 64 * nwin / 2**20, 1)},
        "checks": {"result_matches_cpu_oracle": ok, "all_checks_pass": bool(ok_all)},
        "e2e": {"value": e2e_value, "unit": "points/s", "h2d_bytes_per_step": N_PTS * 32, "d2h_bytes_per_step": 128 * max(wb, 1),
                "ms_per_step": msm_e2e_ms / args.steps},
        "gpu_launches": int(launches_total),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": "k_accumulate (bucket accumulation)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": msm_traffic, "peak_source": peak_src, "kernel_ms": acc_ms,
                     "algorithmic_bytes": MSM_BYTES_PER_POINT * N_PTS,
                     "note": "MSM is integer-ALU bound: 96 B/point of compulsory traffic vs ~16 mixed additions (~190 modular multiplications) per point; "
                             "the accumulation kernel gathers 64 B per (point, window) from the resident table, which is what `traffic` shows",
                     "stage_ms": stages},
        "cpu_baseline": {"value": N_PTS / cpu_msm_s, "unit": "points/s", "cores": threads, "kind": "port",
                         "sample": f"{cpu_reps} x the same 2^16-point MSM (oracle: ark-style Pippenger, 2-way split, best of 8..{orc.host_threads()} threads = {threads}), {cpu_msm_s * 1e3:.1f} ms each"},
        "ntt": {
            "metric": "fp_ntt_elements_per_s", "workload": "2^16-element Fp forward NTT (Radix2EvaluationDomain::fft_in_place)" + ("" if world == 1 else f", {world} replicas"),
            "value": world * N_PTS / (ntt_ms / args.steps * 1e-3), "unit": "elements/s", "ms_per_step": ntt_ms / args.steps,
            "e2e": {"value": world * N_PTS / (ntt_e2e_ms / args.steps * 1e-3), "unit": "elements/s", "h2d_bytes_per_step": N_PTS * 32, "d2h_bytes_per_step": N_PTS * 32},
            "roofline": {"bound": "hbm", "kernel": "k_ntt_pass x2", "achieved": ntt_ach, "peak": peak, "unit": "GB/s", "frac": ntt_ach / peak, "traffic": ntt_traffic, "kernel_ms": ntt_k,
                         "algorithmic_bytes": NTT_BYTES_PER_ELEM * N_PTS},
            "cpu_baseline": {"value": N_PTS / cpu_ntt_s, "unit": "elements/s", "cores": threads, "kind": "port", "sample": f"{cpu_ntt_reps} x the same transform"},
        },
        "extra": extra,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, zk.jacobian_to_affine(zk.PALLAS, result), last["ntt"])
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    if not ok_all:
        # a timed result that differs from the CPU oracle is not a measurement
        print("bench.py: a timed result differs from the CPU oracle", file=sys.stderr)
        sys.exit(3)


if __name__ == "__main__":
    main()
