#!/usr/bin/env python
"""bench.py - contact-force QPs solved per second (BASELINE.json metric).

Workload = BASELINE config C3: the fused FK + Jacobian + QP + J^T f torque pipeline on 2^20 randomised
states per GPU, FP64 (weak scaling: every rank owns its own 2^20-state slice of the counter-based
synthetic batch; no collective on the solve path, one tiny NCCL all-reduce of statistics at the end).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Prints ONE JSON line (rank 0).  `value` = whole-job QP/s with inputs resident in HBM; `e2e` = the same
through the C ABI's host-pointer entry (pinned host buffers, H2D + D2H inside the timed region);
`roofline` = algorithmic FP64 FLOP/s of the fused kernel against the FP64 FMA peak measured on the box;
`cpu_baseline` = the reference's own QuadProg++ (oracle/_ref) or the oracle port on the host cores.
--impl reference times that CPU path alone.
--dump-outputs DIR also writes what the timed solve call returned in its last step (grf, tau, netwrench, flags of
rank 0's slice) as DIR/<name>.npy; the inputs are the same on every run with the same arguments, so two builds can
be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "contact-force QPs solved/sec"
UNIT = "QP/s"
BATCH_PER_GPU = 1 << 20
MODEL = "quadruped_model"   # the URDF the reference's kinematics class actually loads (quadrupedkinematics.cpp:21)
# fixed accounting constants of SURVEY.md 8d: algorithmic FP64 FLOP per QP by stance count
FLOP_PER_QP = {0: 0.0, 1: 6000.0, 2: 12000.0, 3: 21000.0, 4: 30000.0}
WORKLOAD = ("C3: fused FK+Jacobian+QP+J^T.f torque pipeline, 2^20 randomised states per GPU "
            "(60% four-stance, 25% diagonal pairs, 15% three-stance), FP64, model quadruped_model.urdf")




def bench_config(B: int, world: int) -> dict:
    """The `config` object of the JSON line; identical for the GPU arm and the reference arm."""
    bytes_per_qp = ((12 + 4 + 6 + 4) * 8 + 1) + ((12 + 12 + 6) * 8 + 4)
    return {"workload": WORKLOAD, "states_per_gpu": B, "global_batch": world * B,
            "parallelism": f"instance-sharded x{world}, no data-path collective",
            "l2_policy": f"inputs+outputs {B * bytes_per_qp / 1e6:.0f} MB per step exceed the 126 MB L2"}


NCU_RECORD = os.path.join(ROOT, "profiles", "r2_final_ncu.json")   # written by tools/ncu_summary.py from the committed capture
DUMP_STATES = 1 << 17   # states written by --dump-outputs: 31 FP64 values each, 32.5 MB in all


def dump_outputs(out_dir: str, outputs: dict) -> None:
    """Write the [C, B] device outputs of one solve call as out_dir/<name>.npy in float64 (flags too: every uint32 is
    exact there).  A batch larger than DUMP_STATES is sampled: the same seeded, sorted state indices for a given batch
    size on every run."""
    import torch
    B = outputs["flags"].shape[-1]
    idx = np.arange(B) if B <= DUMP_STATES else np.sort(np.random.default_rng(0).choice(B, DUMP_STATES, replace=False))
    sel = torch.from_numpy(idx).to(outputs["flags"].device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        a = t.index_select(-1, sel).cpu().numpy()
        if name == "flags":
            a = a.view(np.uint32)
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


_JSON_FD = None   # the process's real stdout once emit_only_json_on_stdout() has moved fd 1 to stderr


def emit_only_json_on_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too - NCCL writes its version line to stdout at
    NCCL_DEBUG=VERSION, a level at which it ignores NCCL_DEBUG_FILE - so fd 1 is pointed at stderr for the rest of the
    process (nothing is hidden, the NCCL_DEBUG level is the caller's) and the JSON line goes out through the saved fd."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def print_json_line(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, data)


def load_ncu_record():
    """DRAM traffic and executed-pipe figures of one solve call on 2^20 C3 states, from the committed ncu capture
    (a run under the profiler is never a bench value; the bench reports these next to its own timing)."""
    try:
        with open(NCU_RECORD) as f:
            return json.load(f)
    except Exception:
        return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "power_w_max": float(max(power)),
                "samples": len(sm), "reasons": sorted(reasons)}


def pin_to_gpu_numa_node(index: int):
    """Run this process on the CPU cores next to GPU `index` (NVML's ideal affinity) so that the pinned host
    buffers of the end-to-end path are first-touched on that NUMA node; with one process per GPU and the default
    scheduler the eight ranks of a box otherwise share one socket's memory controllers.  Returns the previous
    affinity (restored before the CPU baseline runs) or None."""
    try:
        import pynvml
        prev = os.sched_getaffinity(0)
        pynvml.nvmlInit()
        try:    # CUDA_VISIBLE_DEVICES may renumber the devices: go through the UUID of the CUDA device
            import torch
            handle = pynvml.nvmlDeviceGetHandleByUUID("GPU-" + str(torch.cuda.get_device_properties(index).uuid))
        except Exception:
            handle = pynvml.nvmlDeviceGetHandleByIndex(index)
        pynvml.nvmlDeviceSetCpuAffinity(handle)
        return prev
    except Exception:
        return None


def cpu_reference(st, steps: int, warmup: int, sample: int):
    """The reference's CPU implementation of the path on the host cores: QP assembly per
    ContactForceDistribution.cpp + the reference's own QuadProg++ (oracle/_ref) when it was built,
    else the oracle port.  Returns (QP/s, dict)."""
    from oracle import oracle as O
    from quadruped_locomotion_b200 import legmodel
    M = O.model_array(legmodel.load_model(MODEL))
    kind = "reference" if O.have_ref() else "port"
    solver = O.SOLVER_REF if kind == "reference" else O.SOLVER_GI
    cores = os.cpu_count() or 1
    sub = {k: np.ascontiguousarray(v[..., :sample]) for k, v in st.items()}

    def run(nsolves):
        t0 = time.perf_counter()
        O.solve_wrench_batch(M, sub["q"], sub["quat"], sub["wrench"], sub["mask"], mu=sub["mu"], normals=None,
                             solver=solver, nsolves=nsolves, threads=cores)
        return time.perf_counter() - t0

    for _ in range(max(1, warmup)):
        run(1)
    times = [run(1) for _ in range(max(1, steps))]
    t1 = float(np.mean(times))
    t2 = run(2) if kind == "port" else 2.0 * t1   # the reference solves twice per tick (CFD.cpp:367,120)
    info = {"value": sample / t1, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"first {sample} states of the same workload, {max(1, steps)} passes, one solve per state; "
                      f"solver = {'reference QuadProg++ (qp_solver/src/QuadProg++.cc compiled in place)' if kind == 'reference' else 'oracle Goldfarb-Idnani port'}; "
                      "real OOQP+MA27 is not vendored and cannot run here",
            "value_two_solves_per_state": sample / t2, "ms_per_pass": t1 * 1e3}
    return sample / t1, info


def run_sweep(args, rank, local_rank, world, dev, warmup):
    """BASELINE config C5: the Monte-Carlo robustness sweep (2^14 nominal states x 2^10 perturbations of base attitude,
    friction and wrench scale), sharded by instance over the ranks.  The states are GENERATED ON THE DEVICE
    (qlb_generate_states, bit-identical to synth.make_states), solved, and reduced to qlb_stats on the device: one step
    moves nothing over PCIe but 248 bytes of statistics, and the ranks exchange nothing but those (NCCL all-reduce).
    `value` = solve only (states resident); `e2e` = generate + solve + statistics + all-reduce per step."""
    import torch
    import torch.distributed as dist
    from quadruped_locomotion_b200 import capi, dist as qdist
    B = args.batch if args.batch != BATCH_PER_GPU else (1 << 21)
    solver = capi.Solver(MODEL, device=local_rank)
    stream = torch.cuda.current_stream()
    f64 = lambda n: torch.empty((n, B), dtype=torch.float64, device=dev)  # noqa: E731
    q, quat, wrench, mu, grf, tau, net = f64(12), f64(4), f64(6), f64(4), f64(12), f64(12), f64(6)
    mask = torch.empty(B, dtype=torch.uint8, device=dev)
    flags = torch.empty(B, dtype=torch.int32, device=dev)

    def generate():
        solver.generate_states("C5", B, start=rank * B, q=q, quat=quat, wrench=wrench, mask=mask, mu=mu, stream=stream.cuda_stream)

    def solve():
        solver.solve_wrench(q, quat, wrench, mask, mu, None, grf, tau, flags, net, stream=stream.cuda_stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record(stream)
        for _ in range(steps):
            fn()
        ev1.record(stream)
        barrier()
        t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps

    generate()
    for _ in range(warmup):
        solve()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    launches0 = solver.launches
    ms_step = timed(solve, args.steps)
    launches = solver.launches - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"grf": grf, "tau": tau, "netwrench": net, "flags": flags})
    ms_gen = timed(generate, max(3, args.steps // 4))

    stats_holder = {}

    def sweep_step():
        generate()
        solve()
        s = torch.from_numpy(solver.batch_stats(flags, wrench, net, stream=stream.cuda_stream)).to(dev)
        qdist.allreduce_stats(s)
        stats_holder["s"] = s.cpu().numpy()

    for _ in range(2):
        sweep_step()
    barrier()
    e2e_steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        sweep_step()
    torch.cuda.synchronize()
    t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    sd = qdist.stats_dict(stats_holder["s"])
    if rank == 0:
        line = {
            "metric": METRIC, "value": world * B / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic (generated on the device)",
            "config": {"workload": "C5: Monte-Carlo robustness sweep, perturbed base attitude / friction / wrench scale, "
                                   f"{world * B} samples, FP64, model quadruped_model.urdf", "states_per_gpu": B,
                       "global_batch": world * B, "parallelism": f"instance-sharded x{world}, no data-path collective",
                       "l2_policy": "inputs+outputs exceed the 126 MB L2"},
            "clocks": clocks,
            "e2e": {"value": world * B * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": capi.STATS_NUM * 8, "steps": e2e_steps,
                    "api": "qlb_generate_states + qlb_solve_wrench + qlb_batch_stats + all-reduce of the statistics: nothing "
                           "but 248 bytes per rank leaves the device"},
            "gpu_launches": int(launches), "generate_ms_per_step": ms_gen,
            "stats": {"count": sd["count"], "ok": sd["ok"], "infeasible": sd["infeasible"], "bad_input": sd["bad_input"],
                      "max_iter": sd["max_iter"], "mean_solver_rounds": sd["mean_iterations"],
                      "max_solver_rounds": sd["max_iterations"], "mean_wrench_err": sd["mean_wrench_err"],
                      "max_wrench_err": sd["max_wrench_err"], "active_row_hist": sd["active_hist"]},
        }
        print_json_line(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU, help="states per GPU (default 2^20)")
    ap.add_argument("--config", default="C3")
    ap.add_argument("--cpu-sample", type=int, default=1 << 19)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help=f"write the outputs of the last timed step as DIR/<name>.npy (a fixed sample of {DUMP_STATES} states "
                         "when the batch is larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    warmup = max(3, args.warmup)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    from quadruped_locomotion_b200 import synth
    B = args.batch

    if args.impl == "reference":
        if rank != 0:
            return
        # the same workload as the GPU arm: every step is one pass over the full 2^20-state batch of rank 0
        st = synth.make_states(args.config, B)
        sample = st["q"].shape[1]
        v, info = cpu_reference(st, args.steps, min(warmup, 3), sample)
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": warmup, "ms_per_step": info["ms_per_pass"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "config": bench_config(B, args.gpus),
                "cpu_baseline": info, "gpu_launches": 0,
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print_json_line(line)
        return

    import torch
    import torch.distributed as dist
    from quadruped_locomotion_b200 import capi, dist as qdist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    prev_affinity = pin_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # the contract is ONE JSON line on stdout: NCCL's log (whatever NCCL_DEBUG level the caller chose) goes to
        # stderr, the level itself is left alone so that the communicator lines stay visible to the caller
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        emit_only_json_on_stdout()
        dist.init_process_group("nccl", device_id=dev)

    if args.config.upper() == "C5":
        run_sweep(args, rank, local_rank, world, dev, warmup)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- inputs: this rank's contiguous slice of the global synthetic batch (no inter-GPU traffic)
    st = synth.make_states(args.config, B, start=rank * B)
    keys = ("q", "quat", "wrench", "mask", "mu")
    d = {k: torch.from_numpy(np.ascontiguousarray(st[k])).to(dev) for k in keys}
    grf = torch.empty((12, B), dtype=torch.float64, device=dev)
    tau = torch.empty_like(grf)
    net = torch.empty((6, B), dtype=torch.float64, device=dev)
    flags = torch.empty(B, dtype=torch.int32, device=dev)
    solver = capi.Solver(MODEL, device=local_rank, max_batch=B)
    stream = torch.cuda.current_stream()

    def step():
        solver.solve_wrench(d["q"], d["quat"], d["wrench"], d["mask"], d["mu"], None, grf, tau, flags, net,
                            stream=stream.cuda_stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    fp64_peak = solver.measure_fp64_peak()
    for _ in range(warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    launches0 = solver.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    launches = solver.launches - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"grf": grf, "tau": tau, "netwrench": net, "flags": flags})
    ms_total = ev0.elapsed_time(ev1)
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / args.steps

    # ---- statistics: device reduction + the only collective of the design (NCCL all-reduce, ~240 B)
    stats = torch.from_numpy(solver.batch_stats(flags, d["wrench"], net, stream=stream.cuda_stream)).to(dev)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    qdist.allreduce_stats(stats)
    torch.cuda.synchronize()
    allreduce_ms = (time.perf_counter() - t0) * 1e3
    sd = qdist.stats_dict(stats.cpu().numpy())

    # ---- end to end through the C ABI host entry: pinned host buffers, H2D + D2H inside the timed region
    h = {k: torch.from_numpy(np.ascontiguousarray(st[k])).pin_memory() for k in keys}
    h_grf = torch.empty((12, B), dtype=torch.float64).pin_memory()
    h_tau = torch.empty((12, B), dtype=torch.float64).pin_memory()
    h_net = torch.empty((6, B), dtype=torch.float64).pin_memory()
    h_flags = torch.empty(B, dtype=torch.int32).pin_memory()

    def e2e_step():
        solver.solve_wrench_host(h["q"], h["quat"], h["wrench"], h["mask"], h["mu"], None, h_grf, h_tau, h_flags, h_net)

    e2e_steps = max(3, min(args.steps, 10))

    def time_host(fn):
        """Wall time of e2e_steps calls of a host-pointer entry (each call synchronises), max over ranks."""
        for _ in range(2):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            fn()
        torch.cuda.synchronize()
        tt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    e2e_s = time_host(e2e_step)
    h2d = B * ((12 + 4 + 6 + 4) * 8 + 1)
    d2h = B * ((12 + 12 + 6) * 8 + 4)
    # the e2e result must be the device result
    assert torch.equal(h_grf, grf.cpu()) and torch.equal(h_flags, flags.cpu())

    # the same through the array-of-structs entry: one contiguous block per direction and chunk
    rec_np = capi.wrench_records(st)
    h_rec = torch.from_numpy(rec_np.view(np.uint8).reshape(-1)).pin_memory()
    h_res = torch.empty(B * capi.RESULT_RECORD_DTYPE.itemsize, dtype=torch.uint8).pin_memory()

    def e2e_rec_step():
        solver.solve_records_host(h_rec, h_res)

    e2e_rec_s = time_host(e2e_rec_step)
    res_np = h_res.numpy().view(capi.RESULT_RECORD_DTYPE)
    assert np.array_equal(res_np["grf"].T, h_grf.numpy()) and np.array_equal(res_np["flags"], h_flags.numpy().view(np.uint32))
    h2d_rec, d2h_rec = B * capi.WRENCH_RECORD_DTYPE.itemsize, B * capi.RESULT_RECORD_DTYPE.itemsize
    e2e_soa = {"value": world * B * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "steps": e2e_steps, "api": "qlb_solve_wrench_host (SoA arrays in pinned host memory, copies inside the timed region)"}
    e2e_aos = {"value": world * B * e2e_steps / e2e_rec_s, "unit": UNIT, "h2d_bytes_per_step": h2d_rec,
               "d2h_bytes_per_step": d2h_rec, "steps": e2e_steps,
               "api": "qlb_solve_records_host (qlb_wrench_record[] / qlb_result_record[] in pinned host memory, one 1-D copy per "
                      "chunk and direction, copies inside the timed region)"}
    e2e_best, e2e_other = (e2e_aos, e2e_soa) if e2e_aos["value"] >= e2e_soa["value"] else (e2e_soa, e2e_aos)
    e2e_best = dict(e2e_best, other_entry=e2e_other)

    # ---- the FP32 twin (BASELINE config C4) on the same states: device-resident and end to end
    d32 = {k: (v.float() if v.dtype == torch.float64 else v) for k, v in d.items()}
    grf32 = torch.empty((12, B), dtype=torch.float32, device=dev)
    tau32 = torch.empty_like(grf32)
    net32 = torch.empty((6, B), dtype=torch.float32, device=dev)
    flags32 = torch.empty(B, dtype=torch.int32, device=dev)

    def step32():
        solver.solve_wrench(d32["q"], d32["quat"], d32["wrench"], d32["mask"], d32["mu"], None, grf32, tau32, flags32,
                            net32, stream=stream.cuda_stream)

    for _ in range(warmup):
        step32()
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        step32()
    ev1.record(stream)
    barrier()
    t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step32 = float(t.item()) / args.steps
    h32 = {k: (v.float().pin_memory() if v.dtype == torch.float64 else v) for k, v in h.items()}
    h_grf32 = torch.empty((12, B), dtype=torch.float32).pin_memory()
    h_tau32 = torch.empty((12, B), dtype=torch.float32).pin_memory()
    h_net32 = torch.empty((6, B), dtype=torch.float32).pin_memory()

    def e2e_step32():
        solver.solve_wrench_host(h32["q"], h32["quat"], h32["wrench"], h32["mask"], h32["mu"], None, h_grf32, h_tau32,
                                 h_flags, h_net32)

    e2e_s32 = time_host(e2e_step32)
    f32_err = float(((grf32.double() - grf).abs().amax(0) / grf.abs().amax(0).clamp(min=1.0)).median().item())

    clocks = sampler.stop() if rank == 0 else None

    # ---- roofline: FP64 pipe (SURVEY.md 8d: not HBM-, not tensor-bound), algorithmic FLOP by stance count
    ns = np.array([bin(int(m)).count("1") for m in range(16)])[st["mask"]]
    flop_local = float(sum(FLOP_PER_QP[int(k)] * int((ns == k).sum()) for k in range(5)))
    ft = torch.tensor([flop_local], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ft, op=dist.ReduceOp.SUM)
    flop_total = float(ft.item())
    peaks, peak_src = load_peaks()
    achieved_tf = flop_local / (ms_step * 1e-3) * 1e-12       # per GPU (the kernel of this rank)
    bytes_per_qp = ((12 + 4 + 6 + 4) * 8 + 1) + ((12 + 12 + 6) * 8 + 4)
    hbm_gbs = B * bytes_per_qp / (ms_step * 1e-3) * 1e-9

    if rank == 0:
        value = world * B / (ms_step * 1e-3)
        cpu_v, cpu_info = (None, None)
        if world == 1:
            if prev_affinity is not None:
                os.sched_setaffinity(0, prev_affinity)   # the CPU baseline gets every host core
            cpu_v, cpu_info = cpu_reference(st, 3, 1, min(B, args.cpu_sample))
        rec = load_ncu_record()
        tw = (rec or {}).get("time_weighted") or {}
        roofline = {
            "bound": "fp64", "achieved": achieved_tf, "peak": fp64_peak, "unit": "TFLOP/s",
            "frac": achieved_tf / fp64_peak if fp64_peak > 0 else None,
            "traffic": tw.get("dram_bytes") * (B / float(1 << 20)) if tw.get("dram_bytes") else None,
            "kernel": "one solve call = qlb_single_kernel<double,double,0,2,true> (TMA-staged inputs, kinematics, QP data, "
                      "unconstrained minimiser, active-set rounds from a shared-memory stash) + qlb_quad_kernel<..,2> "
                      "(interior-point fallback, normally an empty list)",
            "note": "frac is ALGORITHMIC: FP64 FLOP by the fixed accounting of SURVEY 8d (30k/21k/12k per 4/3/2-stance QP, an "
                    "eight-iteration interior point) / CUDA-event time of the call, per GPU, over the DFMA peak measured in this "
                    "run (qlb_measure_fp64_peak).  The kernels execute far fewer FLOP than that accounting assumes, so read it as "
                    "throughput relative to an ideal interior-point implementation; `executed` is what the hardware did.",
            "executed": {
                "source": os.path.relpath(NCU_RECORD, ROOT) if rec else None,
                "what": "ncu --set full capture of the same solve call on 2^20 C3 states (profiled run, not this one), "
                        "time-weighted over the launches of the call",
                "fp64_pipe_active_pct_of_elapsed": tw.get("fp64_pipe_elapsed_pct"),
                "fp64_pipe_active_pct_of_active": tw.get("fp64_pipe_active_pct"),
                "issue_active_pct": tw.get("issue_active_pct"),
                "kernels": [{k: kk.get(k) for k in ("name", "time_s", "dram_bytes", "fp64_pipe_elapsed_pct", "issue_active_pct",
                                                     "warps_active_pct", "registers")} for kk in (rec or {}).get("kernels", [])],
            },
            "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of the launches of one solve call from the same capture, "
                            "scaled by states / 2^20; algorithmic bytes are 453 per QP",
            "hbm": {"achieved": hbm_gbs, "peak": peaks.get("hbm_gbs"), "unit": "GB/s",
                    "frac": hbm_gbs / peaks.get("hbm_gbs", 6650.0), "peak_source": peak_src, "bytes_per_qp": bytes_per_qp},
        }
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": bench_config(B, world),
            "clocks": clocks,
            "e2e": e2e_best,
            "gpu_launches": int(launches),
            "roofline": roofline,
            "cpu_baseline": cpu_info,
            "f32": {"value": world * B / (ms_step32 * 1e-3), "unit": UNIT, "ms_per_step": ms_step32,
                    "e2e": {"value": world * B * e2e_steps / e2e_s32, "unit": UNIT,
                            "h2d_bytes_per_step": B * ((12 + 4 + 6 + 4) * 4 + 1), "d2h_bytes_per_step": B * ((12 + 12 + 6) * 4 + 4)},
                    "median_rel_force_diff_vs_f64": f32_err,
                    "note": "qlb_solve_wrench_f32[_host], default core: FP32 arrays and leg kinematics, friction frame + QP in FP64; "
                            "stated tolerance in include/qlb.h and tests/test_gpu_parity.py"},
            "stats": {"ok": sd["ok"], "max_iter": sd["max_iter"], "unverified": sd["unverified"],
                      "mean_solver_rounds": sd["mean_iterations"], "max_solver_rounds": sd["max_iterations"],
                      "mean_wrench_err": sd["mean_wrench_err"], "allreduce_ms": allreduce_ms,
                      "algorithmic_flop_total": flop_total},
        }
        print_json_line(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
