#!/usr/bin/env python3
"""A/B of the MSM launch shell (option msm_pdl): kernels after the first by programmatic dependent launch with no per-call memsets
(1) against plain launches behind two memsets (0).  Workloads: the bench.py headline (2^16-point Pallas MSM on the fixture
generators, scalars splitmix64_limbs(1, 2^16), table window 16, device-resident scalars), cfg1 (its first 2^11 points, library
window) and one zk_msm_batch of 15 x 2^12 scalars against the headline table (host scalars, so the H2D copy is in both arms).
The 256 MiB L2 flush of bench.py runs before every step, outside the timed span.  The two shells alternate in rounds of `--steps`
steps; every step's affine point must equal the first one.  Writes OUT/msm_shell_ab.json and OUT/r03_msm_shell.md (card name and
power limit read in the same run, torch.profiler launch list of one step per shell)."""
import argparse, json, os, subprocess, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import srs_fixture
import proof_systems_b200 as zk
from bench import splitmix64_limbs

ap = argparse.ArgumentParser()
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--out", required=True, help="directory for msm_shell_ab.json and r03_msm_shell.md")
args = ap.parse_args()
os.makedirs(args.out, exist_ok=True)

card = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
ctx = zk.Context(0)
stream = torch.cuda.Stream(); ctx.set_stream(stream.cuda_stream)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
g = ctx.decompress_points(zk.PALLAS, srs_fixture.load("pallas")["g_cmp"])
N = 1 << 16
scalars = splitmix64_limbs(1, N)
d_sc = torch.from_numpy(scalars.view(np.int64)).cuda()
b16 = ctx.upload_bases(zk.PALLAS, g, window_bits=16)
b11 = ctx.upload_bases(zk.PALLAS, g[:1 << 11], window_bits=-1)
batch_sc = splitmix64_limbs(9, 15 << 12).reshape(15, 1 << 12, 4)
workloads = {
    "headline_2^16_w16": (lambda: ctx.msm_dev(b16, d_sc.data_ptr(), N), lambda r: zk.jacobian_to_affine(zk.PALLAS, r)),
    "cfg1_2^11_w-1": (lambda: ctx.msm_dev(b11, d_sc.data_ptr(), 1 << 11), lambda r: zk.jacobian_to_affine(zk.PALLAS, r)),
    "batch15_2^12_w16": (lambda: ctx.msm_batch(b16, batch_sc), lambda r: np.stack([zk.jacobian_to_affine(zk.PALLAS, x) for x in r])),
}


def step(fn):
    flush.fill_(1); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream); r = fn(); e1.record(stream); e1.synchronize()
    return e0.elapsed_time(e1), r


def launch_list(fn):
    """kernels of one step under torch.profiler: name, duration, gap to the previous kernel's end (us)"""
    from torch.profiler import ProfilerActivity, profile
    flush.fill_(1); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn(); torch.cuda.synchronize()
    ks = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "Fill" not in e.name),
                key=lambda e: e.time_range.start)
    rows, prev = [], None
    for e in ks:
        rows.append({"kernel": e.name[:60], "us": round(e.time_range.end - e.time_range.start, 1),
                     "gap_us": None if prev is None else round(e.time_range.start - prev, 1)})
        prev = e.time_range.end
    return rows


report = {"card": card, "rounds": args.rounds, "steps_per_round": args.steps, "workloads": {}}
for name, (fn, affine) in workloads.items():
    times = {0: [], 1: []}
    ref, same = None, True
    for pdl in (1, 0, 1):                      # warm-up of both shells
        ctx.set_option("msm_pdl", pdl)
        for _ in range(3):
            step(fn)
    for rnd in range(args.rounds):
        for pdl in ((1, 0) if rnd % 2 == 0 else (0, 1)):
            ctx.set_option("msm_pdl", pdl)
            for _ in range(args.steps):
                ms, r = step(fn)
                a = affine(r)
                ref = a if ref is None else ref
                same &= bool(np.array_equal(a, ref))
                times[pdl].append(ms)
    w = {"same_affine_every_step": same}
    for pdl, label in ((0, "plain"), (1, "pdl")):
        t = np.array(times[pdl])
        l0 = ctx.launch_count
        ctx.set_option("msm_pdl", pdl)
        fn()
        w[label] = {"median_ms": round(float(np.median(t)), 4), "p10_ms": round(float(np.percentile(t, 10)), 4),
                    "p90_ms": round(float(np.percentile(t, 90)), 4), "steps": int(t.size), "launches_per_call": ctx.launch_count - l0}
        try:
            w[label]["profiler"] = launch_list(fn)
        except Exception as ex:                 # the profiler is optional: the event timings above are the measurement
            w[label]["profiler"] = f"unavailable: {ex!r}"
    w["gain_pct"] = round(100 * (1 - w["pdl"]["median_ms"] / w["plain"]["median_ms"]), 2)
    report["workloads"][name] = w
    print(name, {k: v for k, v in w.items() if k not in ("plain", "pdl")},
          {l: {k: v for k, v in w[l].items() if k != "profiler"} for l in ("plain", "pdl")}, flush=True)
ctx.set_option("msm_pdl", 1)
json.dump(report, open(os.path.join(args.out, "msm_shell_ab.json"), "w"), indent=1)

md = [f"# MSM launch shell A/B (tools/msm_shell_ab.py): plain launches + 2 memsets vs programmatic dependent launch", "",
      f"Card: {card} (name, power limit, max SM clock; read in the same run).  {args.rounds} alternating rounds x {args.steps} steps "
      "per shell, 256 MiB L2 flush before every step (outside the span), CUDA events around each call.", "",
      "| workload | plain median ms (p10-p90) | pdl median ms (p10-p90) | gain | launches | same point every step |", "|---|---|---|---:|---|---|"]
for name, w in report["workloads"].items():
    p, q = w["plain"], w["pdl"]
    md.append(f"| {name} | {p['median_ms']} ({p['p10_ms']}-{p['p90_ms']}) | {q['median_ms']} ({q['p10_ms']}-{q['p90_ms']}) | {w['gain_pct']} % | "
              f"{p['launches_per_call']} / {q['launches_per_call']} | {w['same_affine_every_step']} |")
for name, w in report["workloads"].items():
    for label in ("plain", "pdl"):
        prof = w[label]["profiler"]
        md += ["", f"## {name}, {label}: torch.profiler launch list of one step", ""]
        if isinstance(prof, str):
            md.append(prof)
            continue
        md += ["| kernel | us | gap to previous us |", "|---|---:|---:|"]
        md += [f"| `{r['kernel']}` | {r['us']} | {'' if r['gap_us'] is None else r['gap_us']} |" for r in prof]
open(os.path.join(args.out, "r03_msm_shell.md"), "w").write("\n".join(md) + "\n")
print(json.dumps({k: {"plain": v["plain"]["median_ms"], "pdl": v["pdl"]["median_ms"], "gain_pct": v["gain_pct"], "same": v["same_affine_every_step"]}
                  for k, v in report["workloads"].items()}))
