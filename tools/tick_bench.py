#!/usr/bin/env python
"""Throughput of the controller tick (qlb_controller_update): robot-ticks per second for B robots, device-resident, timed
with CUDA events after warm-up; per-kernel times from a separate torch.profiler run; the latency of a one-robot tick
through the host entry point.  Writes one JSON line per configuration (default profiles/tick_bench.jsonl), each with the
GPU name and power limit read in the same run.  --dtypes float64,float32 adds the same rows for the FP32 twins
(qlb_controller_update_f32[_host]) on the same trot rounded to float32.  Every row names its "dtype", the tick kernels
carry their template argument in the per-kernel times (qlb_tick_epilogue_kernel<double> / <float>), and profiler traces
are named tick_B{B}_{dtype}.pt.trace.json, also with the default --dtypes float64.

Workload: a trot (LF+RH and RF+LH alternate every 8 ticks, robots spread over the 8 phases) with C3-like joint angles and
attitudes, base position / twist noise 0.05, targets 4 mm away, swing gains (300, 250, 400) / (10, 12, 8); 8 input sets
resident on the device, used in turn.  At 2^20 robots the controller state alone (ring of 11 joint-velocity samples) is
1.1 GB, far above the 126 MB L2, so the timed ticks stream from HBM; at 2^14 most of the working set stays in L2."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from quadruped_locomotion_b200 import capi  # noqa: E402

NSETS = 8


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        pl, clk = [x.strip() for x in r.stdout.strip().split(",")]
        info.update(power_limit=pl, max_sm_clock=clk)
    except Exception as e:   # the numbers are still recorded, without the power limit
        info.update(power_limit=f"unavailable ({type(e).__name__})")
    return info


def make_inputs(B, k, dev, g):
    """Tick k of the trot for B robots, generated on the device."""
    off = torch.arange(B, device=dev) % 8
    kk = k + off
    half = (kk // 8) % 2
    ph = (kk % 8).double() / 8.0
    desired = torch.where(half == 0, 5, 10).to(torch.uint8)
    early = ((torch.rand(B, device=dev, generator=g) < 0.3) & (ph > 0.5)).to(torch.uint8) * (15 - desired)
    contact = (desired | early).to(torch.uint8)
    n = lambda *s, sd=1.0: torch.randn(*s, device=dev, dtype=torch.float64, generator=g) * sd  # noqa: E731
    sgn = torch.tensor([1.0, -1.0, 1.0, -1.0], device=dev, dtype=torch.float64)[:, None]
    q = torch.empty((12, B), device=dev, dtype=torch.float64)
    q[0::3] = n(4, B, sd=0.1)
    q[1::3] = sgn * (0.7 + n(4, B, sd=0.1))
    q[2::3] = -sgn * (1.4 + n(4, B, sd=0.15))
    yaw, pitch, roll = n(B, sd=0.3), n(B, sd=0.03), n(B, sd=0.03)
    cy, sy, cp, sp, cr, sr = (torch.cos(0.5 * yaw), torch.sin(0.5 * yaw), torch.cos(0.5 * pitch), torch.sin(0.5 * pitch),
                              torch.cos(0.5 * roll), torch.sin(0.5 * roll))
    quat = torch.stack([cr * cp * cy + sr * sp * sy, sr * cp * cy - cr * sp * sy, cr * sp * cy + sr * cp * sy,
                        cr * cp * sy - sr * sp * cy])
    pos = n(3, B, sd=0.05) + torch.tensor([0.0, 0.0, 0.45], device=dev, dtype=torch.float64)[:, None]
    pose = torch.cat([pos, quat]).contiguous()
    tpose = torch.cat([pos + n(3, B, sd=0.004), quat]).contiguous()
    foot = torch.tensor([0.42, 0.15, -0.4, 0.42, -0.15, -0.4, -0.42, -0.15, -0.4, -0.42, 0.15, -0.4], device=dev,
                        dtype=torch.float64)[:, None]
    return dict(q=q, qd=n(12, B), pose=pose, twist=n(6, B, sd=0.05), tpose=tpose, ttwist=n(6, B, sd=0.05), desired=desired,
                contact=contact, phase=ph.repeat(4, 1).contiguous(), mu=0.4 + 0.6 * torch.rand((4, B), device=dev,
                dtype=torch.float64, generator=g), pt=(foot + n(12, B, sd=0.03)).contiguous(), vt=n(12, B, sd=0.2))


def tick(ctrl, d, out, stream):
    ctrl.update(d["q"], d["qd"], d["pose"], d["twist"], d["tpose"], d["ttwist"], d["desired"], d["contact"], d["phase"],
                out["command"], out["flags"], mu=d["mu"], ptarget=d["pt"], vtarget=d["vt"], grf=out["grf"], stream=stream)


def params():
    p = capi.default_tick_params()
    for c, (kp, kd) in enumerate(((300.0, 10.0), (250.0, 12.0), (400.0, 8.0))):
        p.swing.kp[c] = kp; p.swing.kd[c] = kd
    return p


def cast(d, dtype):
    """The floating-point arrays of an input set in `dtype` (masks unchanged)."""
    return {k: (v.to(dtype).contiguous() if v.is_floating_point() else v) for k, v in d.items()}


ENTRY = {torch.float64: "qlb_controller_update", torch.float32: "qlb_controller_update_f32"}


def bench_device(s, B, ticks, warmup, info, prof_dir, dtype=torch.float64):
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev); g.manual_seed(1234)
    sets = [cast(make_inputs(B, k, dev, g), dtype) for k in range(NSETS)]
    out = dict(command=torch.empty((12, B), dtype=dtype, device=dev), flags=torch.empty(B, dtype=torch.int32, device=dev),
               grf=torch.empty((12, B), dtype=dtype, device=dev))
    ctrl = capi.Controller(s, B, params())
    stream = torch.cuda.current_stream().cuda_stream
    for k in range(warmup):
        tick(ctrl, sets[k % NSETS], out, stream)
    torch.cuda.synchronize()
    l0 = s.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(ticks):
        tick(ctrl, sets[k % NSETS], out, stream)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / ticks
    launches = (s.launches - l0) / ticks
    # the state-mode solve alone on the same inputs (planned stance mask), for comparison
    tau = torch.empty_like(out["grf"])
    for k in range(warmup):
        d = sets[k % NSETS]
        s.solve_state(d["q"], d["pose"], d["twist"], d["tpose"], d["ttwist"], d["desired"], d["mu"], None, out["grf"], tau, out["flags"],
                      stream=stream)
    e0.record()
    for k in range(ticks):
        d = sets[k % NSETS]
        s.solve_state(d["q"], d["pose"], d["twist"], d["tpose"], d["ttwist"], d["desired"], d["mu"], None, out["grf"], tau, out["flags"],
                      stream=stream)
    e1.record()
    torch.cuda.synchronize()
    ms_solve = e0.elapsed_time(e1) / ticks
    # per-kernel device times, separate run under the profiler
    from torch.profiler import ProfilerActivity, profile
    nprof = min(ticks, 10)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(nprof):
            tick(ctrl, sets[k % NSETS], out, stream)
        torch.cuda.synchronize()
    kernels = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0.0)
        if t and ev.key.startswith(("void qlb", "qlb")):
            name = ev.key.split("(")[0].replace("void ", "").replace("qlb::", "")
            kernels[name] = kernels.get(name, 0.0) + t / nprof   # us per tick
    if prof_dir:
        os.makedirs(prof_dir, exist_ok=True)
        prof.export_chrome_trace(os.path.join(prof_dir, f"tick_B{B}_{str(dtype)[6:]}.pt.trace.json"))
    fl = out["flags"].cpu().numpy().view(np.uint32)
    ctrl.close()
    return dict(info, entry=ENTRY[dtype], dtype=str(dtype)[6:], robots=B, ticks=ticks, warmup=warmup, ms_per_tick=ms,
                robot_ticks_per_s=B / ms * 1e3, launches_per_tick=launches, solve_state_ms_same_inputs=ms_solve,
                tick_minus_solve_ms=ms - ms_solve, kernels_us_per_tick=dict(sorted(kernels.items(), key=lambda kv: -kv[1])),
                ok_fraction_last_tick=float(((fl >> 24) & 7 == 0).mean()))


def bench_host(s, ticks, warmup, info, dtype=torch.float64):
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev); g.manual_seed(99)
    sets = [{k: v.cpu().numpy() for k, v in cast(make_inputs(1, k, dev, g), dtype).items()} for k in range(NSETS)]
    ctrl = capi.Controller(s, 1, params())
    npt = np.float32 if dtype == torch.float32 else np.float64
    cmd = np.zeros((12, 1), npt); fl = np.zeros(1, np.uint32); grf = np.zeros((12, 1), npt)
    lat = []
    for k in range(warmup + ticks):
        d = sets[k % NSETS]
        t0 = time.perf_counter()
        ctrl.update_host(d["q"], d["qd"], d["pose"], d["twist"], d["tpose"], d["ttwist"], d["desired"], d["contact"], d["phase"],
                         cmd, fl, mu=d["mu"], ptarget=d["pt"], vtarget=d["vt"], grf=grf)
        if k >= warmup:
            lat.append((time.perf_counter() - t0) * 1e6)
    ctrl.close()
    lat = np.array(lat)
    return dict(info, entry=ENTRY[dtype] + "_host", dtype=str(dtype)[6:], robots=1, ticks=ticks, warmup=warmup, us_median=float(np.median(lat)),
                us_p99=float(np.percentile(lat, 99)), us_max=float(lat.max()), timer="host clock around the call (it synchronises)")


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "tick_bench.jsonl"))
    ap.add_argument("--ticks", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--host-ticks", type=int, default=2000)
    ap.add_argument("--sizes", default="14,20", help="log2 of the robot counts")
    ap.add_argument("--trace-dir", default=None, help="also write the profiler traces there")
    ap.add_argument("--dtypes", default="float64", help="array types of the caller: float64 and/or float32, comma-separated")
    a = ap.parse_args()
    dtypes = [{"float64": torch.float64, "float32": torch.float32}[t.strip()] for t in a.dtypes.split(",")]
    if not torch.cuda.is_available():
        raise SystemExit("tick_bench needs a CUDA device")
    info = gpu_info()
    s = capi.Solver("quadruped_model")
    s.set_limb_dynamics("quadruped_model")
    rows = [bench_device(s, 1 << int(e), a.ticks, a.warmup, info, a.trace_dir, dt) for e in a.sizes.split(",") for dt in dtypes]
    rows += [bench_host(s, a.host_ticks, 100, info, dt) for dt in dtypes]
    s.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for r in rows:
            line = json.dumps(r)
            print(line, flush=True)
            f.write(line + "\n")


if __name__ == "__main__":
    main()
