#!/usr/bin/env python
"""bench.py — GN iterations/sec of the batched 72-joint IK hot path (BASELINE.json metric).

A *step* is one batched solve: every instance of the per-GPU shard runs ``ITERS`` damped Gauss-Newton
iterations (minIterations = maxIterations = ITERS, so no instance stops early) of
FK sweep -> residual/Jacobian -> JtJ/Jtr -> damped Cholesky -> update.

Default workload "cfg3-shard": the per-GPU shard of BASELINE.json configs[2] — the configuration the
metric/target is quoted on ("72-joint / 128-residual batch at 8xB200") — 8192 x humanoid72 with 24
Position + 6 Orientation constraints (m = 126 -> 128 rows, n = 220), constant damping 0.05, weak
scaling (8 GPUs = 65536 instances = cfg3 exactly). ``--workload cfg2`` / ``cfg4`` select the other
single-GPU configs.

    value   : whole-job GN iterations/s with parameters and targets resident in HBM
    e2e     : same metric through mb2_solver_solve with HOST (pinned) buffers: H2D of targets and initial
              parameters and D2H of solved parameters + per-instance results inside the timed region
    roofline: the JtJ kernel (the kernel BASELINE's metric names), algorithmic m*n*(n+1) FLOP per
              instance-iteration over its CUDA-event time, against the measured tensor peak
    cpu_baseline / --impl reference: the oracle restatement of the reference's CPU solver (one solver per
              instance over all host threads, as tensor_ik.cpp:127), bounded sample
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ITERS = 10
WORKLOADS = {
    "cfg3-shard": dict(batch=8192, rig="humanoid72", orientation=True, rows_m=126, params_n=220, global_batch=65536, desc="8192/GPU x humanoid72, 24 Position + 6 Orientation (m=126->128, n=220), lambda=0.05"),
    "cfg2": dict(batch=4096, rig="humanoid72", orientation=False, rows_m=72, params_n=220, desc="4096/GPU x humanoid72, 24 Position (m=72, n=220), lambda=0.05"),
    "cfg5": dict(batch=8192, rig="mixed", orientation=False, rows_m=None, params_n=None, global_batch=65536,
                 desc="8192/GPU mixed rigs: chain22 25% / humanoid72 50% / body150 15% / bodyhands300 10%, Position constraints U{4..200} capped by rig, lambda=0.05"),
    "cfg4": dict(batch=2048, rig="bodyhands300", orientation=False, rows_m=600, params_n=424, global_batch=16384, desc="2048/GPU x bodyhands300, 200 Position (m=600, n=424), lambda=0.05"),
}


def make_problem(workload, batch, seed_offset=0):
    from momentum_b200.problems import bodyhands_problem, humanoid_problem

    w = WORKLOADS[workload]
    if w["rig"] == "humanoid72":
        return humanoid_problem(batch, seed=12347 + seed_offset, orientation=w["orientation"])
    return bodyhands_problem(batch, seed=12349 + seed_offset)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm_gbs=6650.0, bf16=1590.0, bf16_sustained=1400.0, src="fallback")


def measured_traffic(workload, batch):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full captures (profiles/ncu_traffic.json);
    only valid for the exact workload / batch they were captured on."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return {}
    d = json.load(open(p))
    return d.get(f"{workload}:{batch}", {}).get("dram_bytes_per_launch", {})


class ClockSampler:
    """SM clock / clock-event reasons sampled DURING the timed regions (B200_PROFILING.md recipe). NVML is polled in-process
    (the timed regions of the default run are ~45 ms each, shorter than one nvidia-smi start-up) every 25 ms; the two queries take
    microseconds (scripts/nvml_cost.py: median 3 us), --clock-poll-ms changes the period."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown"}

    def __init__(self, index, period_s=0.025):
        self.period_s = period_s
        self.index, self.sm, self.mask, self.max_mhz, self.handle, self.nvml = index, [], 0, None, None, None
        self.stop_flag = threading.Event()
        self.thread = None
        self.error = None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nvml = pynvml
            try:
                uuid = str(torch.cuda.get_device_properties(self.index).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
        except Exception as e:  # noqa: BLE001
            self.error = f"nvml unavailable: {e}"

    def _poll(self):
        nv = self.nvml
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                try:
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                except Exception:
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            except Exception as e:  # noqa: BLE001
                self.error = str(e)
                return
            time.sleep(self.period_s)

    def stop(self):
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [self.error or "nvml unavailable"], "samples": 0}
        self.stop_flag.set()
        self.thread.join(timeout=2)
        reasons = sorted(name for bit, name in self.REASONS.items() if self.mask & bit)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(self.sm)}


def bench_config(args, world):
    """The `config` dict of both arms' JSON lines (the driver compares them key by key): the workload as named in BASELINE.json, never
    anything measured. The CPU arm times a bounded sample of this workload (its size is in cpu_baseline.sample)."""
    w = WORKLOADS[args.workload]
    B = args.batch_per_gpu or w["batch"]
    return {"workload": args.workload, "desc": w["desc"], "batch_per_gpu": B, "global_batch": B * world, "iterations_per_solve": ITERS,
            "rows_m": w["rows_m"], "params_n": w["params_n"], "parallelism": f"dp{world} (instances sharded, no data-path collective)",
            "jtj_mode": args.jtj_mode, "cholesky_mode": args.cholesky_mode, "fused_mode": getattr(args, "fused_mode", 0),
            "l2": "256 MB buffer written between timed steps (L2 flush)"}


def time_cpu_arm(workload, seconds, threads=None):
    """The reference's CPU algorithm (oracle restatement, float, -march=native timing build, one solver per instance over the host
    threads this process may use — affinity mask capped by the cgroup quota — as tensor_ik.cpp:127 does with dispenso) on a bounded
    sample of the workload. Returns (it/s, threads, sample description, single-thread it/s)."""
    from oracle.binding import OracleFunction, hardware_threads

    threads = threads or hardware_threads()
    sample = max(threads * 4, 64)
    ch, efs, theta0, _ = make_problem(workload, sample)
    orc = OracleFunction(ch, efs, "float32", native=True)
    kw = dict(min_iterations=ITERS, max_iterations=ITERS, threshold=1.0, regularization=0.05, final_errors=False)
    orc.solve_batch(theta0, threads=threads, **kw)
    reps, its, t0 = 0, 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        its += int(orc.solve_batch(theta0, threads=threads, **kw)["iterations"].sum())
        reps += 1
    dt = time.perf_counter() - t0
    # single-thread figure on a few instances (SURVEY 8d (ii))
    n1 = min(sample, 8)
    t1 = time.perf_counter()
    its1 = int(orc.solve_batch(theta0[:n1], threads=1, **kw)["iterations"].sum()) if n1 == sample else None
    if its1 is None:
        ch1, efs1, th1, _ = make_problem(workload, n1)
        o1 = OracleFunction(ch1, efs1, "float32", native=True)
        t1 = time.perf_counter()
        its1 = int(o1.solve_batch(th1, threads=1, **kw)["iterations"].sum())
    single = its1 / (time.perf_counter() - t1)
    build = "-O3 -march=native, FMA + reassociation, row-major blocked LLT" if getattr(orc._L, "is_native", False) else "portable x86-64-v3 checker build"
    desc = (f"{reps} x {sample} instances x {ITERS} GN iterations (oracle restatement of the reference solver, float, {build}; one solver per "
            f"instance over {threads} host threads; single thread: {single:.0f} GN it/s)")
    return its / dt, threads, desc, single, sample


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU algorithm (oracle port, float) on the host cores."""
    if rank != 0:
        return
    budget = max(5.0, min(20.0, 2.0 * (args.steps + args.warmup)))  # bounded: the whole run ends within a few minutes whatever K / W are
    t0 = time.perf_counter()
    value, threads, desc, single, sample = time_cpu_arm(args.workload, budget)
    dt = time.perf_counter() - t0
    line = {"impl": "reference", "metric": "GN iterations/sec (batched 72-joint IK)", "value": value, "unit": "GN it/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sample * ITERS / value, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": bench_config(args, world),
            "cpu_baseline": {"value": value, "unit": "GN it/s", "cores": threads, "kind": "port", "sample": desc, "single_thread_value": single},
            "e2e": {"value": value, "unit": "GN it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "wall_s": dt}
    print(json.dumps(line))


def measure_workload(ms, torch, workload, B, rank, local_rank, args, steps, warmup, min_it=ITERS, max_it=ITERS, e2e=True, profile=True, flush=None, barrier=None,
                     keep_outputs=False):
    """Device-resident timing (CUDA events on the launching stream, L2 flushed between steps), the end-to-end leg through mb2_set_targets +
    mb2_solver_solve with pinned host buffers, and one profiling solve (events around every launch + in-kernel phase cycles).
    keep_outputs: out["outputs"] holds what the last timed step returned to its caller (solved parameters + per-instance results)."""
    ch, efs, theta0, _ = make_problem(workload, B, seed_offset=1000 * rank)  # each rank owns a different shard
    n = ch.num_params
    fn = ms.SkeletonSolverFunction(ch, B, efs, device=local_rank)
    fn.upload_targets()
    opts = ms.GaussNewtonSolverOptions(min_iterations=min_it, max_iterations=max_it, threshold=1.0, regularization=0.05, jtj_mode=args.jtj_mode,
                                       cholesky_mode=args.cholesky_mode, fused_mode=args.fused_mode)
    solver = ms.GaussNewtonSolver(opts, fn)
    stream = torch.cuda.current_stream().cuda_stream
    theta0_dev = torch.from_numpy(theta0.astype(np.float32)).cuda()
    theta_dev = torch.empty_like(theta0_dev)

    def device_step():
        theta_dev.copy_(theta0_dev)
        solver.solve_device(theta_dev.data_ptr(), stream)

    for _ in range(warmup):
        device_step()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    total_ms = 0.0
    for _ in range(steps):
        flush.zero_()  # flush L2 between timed iterations
        torch.cuda.synchronize()
        ev0.record()
        device_step()
        ev1.record()
        torch.cuda.synchronize()
        total_ms += ev0.elapsed_time(ev1)
    barrier()
    res = solver.get_results()
    out = {"ch": ch, "efs": efs, "n": n, "B": B, "solver": solver, "fn": fn, "total_ms": total_ms, "its_per_step": int(res["iterations"].sum()),
           "err_sum": float(res["errors"].sum()), "launches": solver.get_counters()[1], "status_bad": int((res["status"] != 0).sum())}
    if keep_outputs:  # before the profiling and end-to-end solves below overwrite theta_dev
        out["outputs"] = {"params": theta_dev.cpu().numpy(), **res}
    if profile:
        solver.set_profiling(1)  # events around the production kernels: the per-kernel times
        device_step()
        torch.cuda.synchronize()
        solver.get_results()
        out["phase_ms"], out["phase_launches"] = solver.get_phase_times()
        solver.set_profiling(2)  # instrumented instantiations: only the phase SHARES are taken from this pass
        device_step()
        torch.cuda.synchronize()
        solver.get_results()
        out["fused"] = solver.get_fused_profile()
        solver.set_profiling(0)
    if e2e:
        theta0_pin = torch.from_numpy(theta0.astype(np.float32)).pin_memory()
        # Two long-lived pinned staging buffers used alternately, as a streaming caller keeps them: mb2_solver_solve uploads the buffer's
        # parameters, solves in place and downloads the result into the same buffer. (Measured alternatives: a FRESH pinned buffer per step
        # makes the 7.2 MB transfers 0.7 - 1.1 ms slower - the DMA path is slow on host pages it has not seen recently: 9.3 - 9.8 instead of
        # 8.66 ms per step; refilling the idle buffer from the host while the device works costs more than it hides - the host memcpy fights
        # the D2H for memory bandwidth and torch's copy threads stall for tens of ms now and then.) From its second use on a buffer holds the
        # previous result of that buffer: with minIterations = maxIterations the work of a step does not depend on the starting point.
        theta_pins = [theta0_pin.clone().pin_memory() for _ in range(2)]
        target_pins = [torch.from_numpy(np.ascontiguousarray(e.targets, np.float32)).pin_memory() for e in efs]
        count = [0]

        def e2e_step():
            buf = theta_pins[count[0] % 2]
            count[0] += 1
            for idx, tp in enumerate(target_pins):
                fn._check(fn._L.mb2_set_targets(fn._h, idx, ms.C.cast(tp.data_ptr(), ms._fp)))
            return solver.solve_host_pointer(buf.data_ptr(), results=True)  # mb2_solver_solve: parameters in / out + per-instance results

        for _ in range(max(2, warmup // 2)):  # (the first call allocates the staging buffers: 20 - 30 ms)
            e2e_step()
        barrier()
        step_s = []
        t0 = time.perf_counter()
        for _ in range(steps):
            t1 = time.perf_counter()
            e2e_step()  # returns after the parameters and the results are on the host (mb2_solver_solve synchronises)
            step_s.append(time.perf_counter() - t1)
        torch.cuda.synchronize()
        out["e2e_s"] = time.perf_counter() - t0
        out["e2e_step_ms"] = [1e3 * x for x in step_s]
        out["h2d"] = int(theta0_pin.numel() * 4 + sum(tp.numel() * 4 for tp in target_pins))
        out["d2h"] = int(theta0_pin.numel() * 4 + B * (8 + 4 + 4))
    return out


DUMP_LIMIT_BYTES = 64 * 2 ** 20


def dump_outputs(directory, outputs, prefix=""):
    """--dump-outputs: what the last timed step returned, one row per instance, as <directory>/<prefix><name>.npy (parameters float32, per-instance
    results float64) so that two builds can be compared output for output. Above DUMP_LIMIT_BYTES in all a fixed seeded sample of the
    instances is written; instance.npy always lists the instances written."""
    arrays = {"params": outputs["params"].astype(np.float32), "errors": outputs["errors"].astype(np.float64),
              "iterations": outputs["iterations"].astype(np.float64), "status": outputs["status"].astype(np.float64)}
    B = arrays["params"].shape[0]
    row_bytes = sum(a[0].nbytes for a in arrays.values()) + 8  # + the instance index
    keep = min(B, (DUMP_LIMIT_BYTES - 4096) // row_bytes)  # 4096: the .npy headers
    idx = np.arange(B) if keep == B else np.sort(np.random.default_rng(0).choice(B, keep, replace=False))
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, prefix + "instance.npy"), idx.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(directory, prefix + name + ".npy"), a[idx])


def kernel_report(m, peaks, workload):
    """Per-kernel roofline entries from the profiling solve. ALGORITHMIC bytes / flops per instance and launch (DESIGN.md section 4)."""
    solver, n, B, efs = m["solver"], m["n"], m["B"], m["efs"]
    st = solver.get_plan_stats()
    tf32_peak = 0.5 * peaks["bf16"]  # TF32 dense = half the bf16 rate (B200_PROFILING.md table); bf16 figure is the measured cuBLAS burst
    hbm_peak = peaks["hbm_gbs"]
    pm, pl = m["phase_ms"], m["phase_launches"]
    sweep_ms = pm[0] / max(1, pl[0]); jtj_ms = pm[1] / max(1, pl[1]); chol_ms = pm[2] / max(1, pl[2])
    m_rows = WORKLOADS[workload]["rows_m"]
    target_floats = sum(int(np.prod(np.asarray(e.targets).shape[1:])) for e in efs)
    traffic = measured_traffic(workload, B)
    jtj_flops = float(m_rows) * n * (n + 1)  # SURVEY 8(d): the JtJ credit, whatever the kernel executes

    def hbm_entry(name, key, bytes_per_instance, ms_):
        ach = bytes_per_instance * B / (ms_ * 1e-3) / 1e9 if ms_ > 0 else 0.0
        return {"kernel": name, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "peak_source": f"{peaks['src']} copy bandwidth",
                "traffic": traffic.get(key), "ms_per_launch": ms_, "algorithmic_bytes_per_instance": bytes_per_instance}

    k1_bytes = 4.0 * (n + target_floats + st["jacobian_nonzeros"] + m_rows) + 8.0
    kernels = [hbm_entry("sweepKernel<true> (three-pass FK + residual + Jacobian strips)", "fk_residual_jacobian", k1_bytes, sweep_ms)]
    fused = m["fused"]
    ntiles = st["cholesky_tiles"]
    gram_flops = 2.0 * st["gram_macs"]
    jtj_phase = None
    if fused["fused"] == 2:  # Gram + Cholesky in one launch: strips in, theta / delta / bookkeeping out; tiles never leave the SM
        gc_bytes = 4.0 * (st["strip_floats"] + 4 * st["normal_parameters"]) + 32.0
        e = hbm_entry("gramCholeskyKernel (tile-sparse J^T J on mma.sync 3xTF32 -> TMEM -> tiles in shared memory -> tile Cholesky + update)", "gram_cholesky", gc_bytes, chol_ms)
        cyc = fused["phase_cycles"]
        tot = float(sum(cyc.values())) or 1.0
        share = (cyc["gram"] + cyc["tiles_from_tmem"]) / tot
        gram_ms = chol_ms * share
        jtj_phase = {"where": "Gram phase of gramCholeskyKernel (in-kernel cycle share x the kernel's event time)", "share_of_kernel": share, "ms": gram_ms}
        e["phase_cycle_shares"] = {k: v / tot for k, v in cyc.items() if v}
        e["phase_cycles_per_launch"] = {k: v / max(1, pl[2]) for k, v in cyc.items() if v}  # SM cycles of one steady-state CTA (block batch / 2), barrier to barrier
        kernels.append(e)
    elif st["strip_floats"] > 0:
        gram_bytes = 4.0 * (st["strip_floats"] + ntiles * 256 + 16 * ((st["normal_parameters"] + 15) // 16))
        kernels.append(hbm_entry("gramTilesKernel (tile-sparse J^T J / J^T r, mma.sync 3xTF32 over non-zero strips)", "jtj_jtr", gram_bytes, jtj_ms))
        k3_bytes = 4.0 * (ntiles * 256 + 4 * st["normal_parameters"])
        kernels.append(hbm_entry("choleskyScheduledKernel (damped LLT + solves + update)", "cholesky_update", k3_bytes, chol_ms))
        jtj_phase = {"where": "gramTilesKernel", "share_of_kernel": 1.0, "ms": jtj_ms}
    else:
        k2_bytes = 4.0 * (m_rows * (st["jacobian_columns"] + 1) + (st["normal_parameters"] + 1) * (st["normal_parameters"] + 2) / 2)
        ach = jtj_flops * B / (jtj_ms * 1e-3) / 1e12 if jtj_ms > 0 else 0.0
        dense = st["jacobian_columns"] + 1 <= 512
        kernels.append({"kernel": "jtjTensorKernel (JtJ/Jtr, tcgen05 3xTF32)" if dense else "jtjSimtKernel", "bound": "tensor", "achieved": ach, "peak": tf32_peak, "unit": "TFLOP/s",
                        "frac": ach / tf32_peak, "peak_source": f"0.5 x {peaks['src']} bf16 cuBLAS burst ({peaks['bf16']} TF/s) = TF32 dense", "traffic": traffic.get("jtj_jtr"),
                        "ms_per_launch": jtj_ms, "algorithmic_flops_per_instance": jtj_flops, "algorithmic_bytes_per_instance": k2_bytes})
        k3_entries = ntiles * 256 if ntiles else st["normal_parameters"] * (st["normal_parameters"] + 1) / 2
        kernels.append(hbm_entry("choleskyScheduledKernel (damped LLT + solves + update)" if ntiles else "choleskyKernel (dense LLT + solves + update)", "cholesky_update",
                                 4.0 * (k3_entries + 4 * st["normal_parameters"]), chol_ms))
    if jtj_phase is not None and jtj_phase["ms"] > 0:
        dense_eq = jtj_flops * B / (jtj_phase["ms"] * 1e-3) / 1e12
        executed = gram_flops * B / (jtj_phase["ms"] * 1e-3) / 1e12
        step_ms = sweep_ms + jtj_ms + chol_ms
        jtj_phase.update({"credited_flops_per_instance": jtj_flops, "credited_tflops": dense_eq, "credited_frac_of_tf32_peak": dense_eq / tf32_peak,
                          "executed_flops_per_instance": gram_flops, "executed_tflops": executed, "executed_frac_of_tf32_peak": executed / tf32_peak,
                          "credited_tflops_end_to_end": jtj_flops * B / (step_ms * 1e-3) / 1e12 if step_ms > 0 else 0.0,
                          "tf32_peak": tf32_peak, "note": "credit = m n (n + 1) per instance-iteration (SURVEY 8d); executed = the multiply-adds of the non-zero 4x16 strips only; "
                                                         "mma.sync (HMMA) path, not tcgen05: see profiles/sass_r02.txt"})
    return kernels, jtj_phase, {"fk_residual_jacobian": sweep_ms, "jtj_jtr": jtj_ms, "cholesky_update": chol_ms}, st


def extra_workloads(ms, torch, args, rank, local_rank, flush, barrier, peaks):
    """Measured in the same run (N = 1 only): the other single-GPU configs, a convergence-mode solve, the persistent kernel at a small
    batch, and the cfg5 mixed-rig batch through the bucketing front end. Compact figures; the headline stays the cfg3 shard."""
    ex = {}
    for wl in ("cfg2", "cfg4"):
        try:
            B = WORKLOADS[wl]["batch"]
            m = measure_workload(ms, torch, wl, B, rank, local_rank, args, steps=3, warmup=3, e2e=False, flush=flush, barrier=barrier)
            kernels, jtj, kms, st = kernel_report(m, peaks, wl)
            ex[wl] = {"desc": WORKLOADS[wl]["desc"], "value": m["its_per_step"] * 3 / (m["total_ms"] * 1e-3), "unit": "GN it/s", "ms_per_step": m["total_ms"] / 3, "batch": B,
                      "kernels_ms_per_iteration": kms, "jtj": jtj, "path": {0: "three kernels", 1: "persistent", 2: "sweep + gramCholesky"}[m["fused"]["fused"]],
                      "tiles": st["cholesky_tiles"], "levels": st["cholesky_levels"], "roofline_all_kernels": kernels}
            del m
        except Exception as e:  # noqa: BLE001
            ex[wl] = {"error": str(e)}
    try:  # convergence mode: SolverOptions min 1 / max 50, threshold 1 (what the parity tests run)
        B = WORKLOADS["cfg3-shard"]["batch"]
        m = measure_workload(ms, torch, "cfg3-shard", B, rank, local_rank, args, steps=2, warmup=2, min_it=1, max_it=50, e2e=False, profile=False, flush=flush, barrier=barrier)
        res = m["solver"].get_results()
        ex["cfg3_convergence_mode"] = {"value": m["its_per_step"] * 2 / (m["total_ms"] * 1e-3), "unit": "GN it/s", "ms_per_solve": m["total_ms"] / 2,
                                       "mean_iterations": float(res["iterations"].mean()), "max_iterations": int(res["iterations"].max()), "min_iterations": int(res["iterations"].min())}
        del m
    except Exception as e:  # noqa: BLE001
        ex["cfg3_convergence_mode"] = {"error": str(e)}
    try:  # one wave of the persistent whole-solve kernel (a latency figure: small batches, single launch, no host round trip)
        small = {}
        for fm, name in ((ms.FUSED_AUTO, "auto"), (ms.FUSED_PERSISTENT, "persistent")):
            a2 = argparse.Namespace(**{**vars(args), "fused_mode": fm})
            m = measure_workload(ms, torch, "cfg3-shard", 256, rank, local_rank, a2, steps=5, warmup=3, e2e=False, profile=False, flush=flush, barrier=barrier)
            small[name] = {"ms_per_solve": m["total_ms"] / 5, "launches": m["launches"]}
            del m
        ex["cfg3_256_instances_latency"] = small
    except Exception as e:  # noqa: BLE001
        ex["cfg3_256_instances_latency"] = {"error": str(e)}
    try:
        ex["cfg5"] = measure_mixed(ms, torch, args, local_rank, WORKLOADS["cfg5"]["batch"], rank)
    except Exception as e:  # noqa: BLE001
        ex["cfg5"] = {"error": str(e)}
    return ex


def measure_mixed(ms, torch, args, local_rank, N, rank, steps=2):
    """cfg5 per-GPU shard through mb2_mixed_batch_solve: host buffers in, host buffers out (an end-to-end figure by construction)."""
    from momentum_b200.problems import mixed_problem

    rigs, inst = mixed_problem(N, seed=12351 + 1000 * rank)
    mb = ms.MixedBatch(device=local_rank)
    rid = {name: mb.add_rig(ch) for name, (ch, _) in rigs.items()}
    for x in inst:
        mb.add_instance(rid[x["rig"]], x["parents"], x["offsets"], x["weights"], x["targets"], x["theta0"])
    st = mb.stats()
    opts = ms.GaussNewtonSolverOptions(min_iterations=ITERS, max_iterations=ITERS, threshold=1.0, regularization=0.05)
    mb.solve(opts)  # builds every bucket's plan (once) and warms up
    for i, x in enumerate(inst):
        mb.set_parameters(i, x["theta0"])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    its = 0
    for _ in range(steps):
        out = mb.solve(opts)
        its += int(out["iterations"].sum())
        for i, x in enumerate(inst):
            mb.set_parameters(i, x["theta0"])
    dt = time.perf_counter() - t0
    per_rig = {}
    for b in range(st["buckets"]):
        info = mb.bucket_info(b)
        name = [k for k, v in rid.items() if v == info["rig"]][0]
        d = per_rig.setdefault(name, {"instances": 0, "buckets": 0, "iterations": 0})
        d["instances"] += info["instances"]; d["buckets"] += 1; d["iterations"] += info["iterations"]
    return {"desc": WORKLOADS["cfg5"]["desc"], "value": its / dt, "unit": "GN it/s (host buffers in and out, bucket staging included)", "instances": N, "buckets": st["buckets"],
            "padding_waste": st["padding_waste"], "largest_bucket": st["largest_bucket"], "per_rig": per_rig, "status_bad": int((out["status"] != 0).sum()), "ms_per_solve": 1e3 * dt / steps}


def measure_sharded(ms, torch, args, B):
    """Single-process multi-GPU (mb2_sharded_solver_*, ik_sharded.cpp): B instances per device, one host thread per shard, host buffers in
    and out (pinned), aggregate on the host. Wall clock around mb2_sharded_solver_solve."""
    N = args.sharded
    ch, efs, theta0, _ = make_problem(args.workload, B * N)
    proto = ms.SkeletonSolverFunction(ch, 1, efs, device=0)  # the definition only: targets go to the shards
    opts = ms.GaussNewtonSolverOptions(min_iterations=ITERS, max_iterations=ITERS, threshold=1.0, regularization=0.05, jtj_mode=args.jtj_mode,
                                       cholesky_mode=args.cholesky_mode, fused_mode=args.fused_mode)
    sh = ms.ShardedGaussNewtonSolver(opts, proto, B * N, list(range(N)), error_functions=efs)
    pins = [torch.from_numpy(theta0.astype(np.float32)).pin_memory() for _ in range(2)]
    for i in range(max(2, args.warmup)):
        sh.solve_host_pointer(pins[i % 2].data_ptr())
    step_ms = []
    t0 = time.perf_counter()
    for i in range(args.steps):
        t1 = time.perf_counter()
        sh.solve_host_pointer(pins[i % 2].data_ptr())
        step_ms.append(round(1e3 * (time.perf_counter() - t1), 3))
    dt = time.perf_counter() - t0
    agg = sh.get_aggregate()
    value = agg["iterations"] * args.steps / dt
    return {"metric": "GN iterations/sec (batched 72-joint IK)", "value": value, "unit": "GN it/s", "n_gpus": N, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "mode": "one process, mb2_sharded_solver_solve over host buffers (end to end by construction)", "config": bench_config(args, N),
            "e2e": {"value": value, "unit": "GN it/s", "h2d_bytes_per_step": int(theta0.size * 4), "d2h_bytes_per_step": int(theta0.size * 4 + B * N * 16), "step_ms": step_ms},
            "aggregate": agg, "shards": sh.shards()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="cfg3-shard", choices=sorted(WORKLOADS))
    ap.add_argument("--batch-per-gpu", type=int, default=0)
    ap.add_argument("--jtj-mode", type=int, default=0)
    ap.add_argument("--cholesky-mode", type=int, default=0)
    ap.add_argument("--fused-mode", type=int, default=0)
    ap.add_argument("--strong", action="store_true", help="strong scaling: the workload's global batch (cfg3: 65536) is split over the ranks")
    ap.add_argument("--sharded", type=int, default=0, help="ONE process driving this many GPUs through mb2_sharded_solver_* (end-to-end figure only; not the driver's torchrun mode)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--clock-poll-ms", type=float, default=25.0, help="NVML clock / throttle-reason sampling period during the timed regions")
    ap.add_argument("--no-extras", action="store_true", help="skip the other workloads measured in the same run (cfg2, cfg4, cfg5, convergence mode)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's solved parameters and per-instance results to "
                    "DIR/<name>.npy (DIR/rank<r>_<name>.npy with several ranks); the inputs are seeded, so runs with the same arguments are comparable")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.sharded > 0 or args.workload == "cfg5"):
        ap.error("--dump-outputs covers the device-resident path of cfg2, cfg3-shard and cfg4")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    from momentum_b200 import solver as ms

    assert torch.cuda.is_available(), "bench.py needs a B200 (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if args.strong:
        total = WORKLOADS[args.workload].get("global_batch", WORKLOADS[args.workload]["batch"] * 8)
        args.batch_per_gpu = total // world
    B = args.batch_per_gpu or WORKLOADS[args.workload]["batch"]
    work_stream = torch.cuda.Stream()  # a real (non-NULL) stream: NULL means "the handle's own stream" in the C-ABI
    torch.cuda.set_stream(work_stream)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    peaks = measured_peaks()
    if args.sharded > 0:
        print(json.dumps(measure_sharded(ms, torch, args, B)))
        return
    if args.workload == "cfg5":
        r = measure_mixed(ms, torch, args, local_rank, B, rank, steps=args.steps)
        from momentum_b200.distributed import aggregate_solve_stats

        its_total, _, _ = aggregate_solve_stats(float(r["value"]), 0.0, 0.0, device="cuda")
        if rank == 0:
            line = {"metric": "GN iterations/sec (mixed-rig batch through the bucketing front end)", "value": its_total, "unit": "GN it/s", "n_gpus": world, "steps": args.steps,
                    "warmup": args.warmup, "ms_per_step": r["ms_per_solve"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                    "config": bench_config(args, world), "cfg5": r, "e2e": {"value": its_total, "unit": "GN it/s", "h2d_bytes_per_step": None, "d2h_bytes_per_step": None}}
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return

    sampler = ClockSampler(local_rank, args.clock_poll_ms * 1e-3)
    sampler.start()
    m = measure_workload(ms, torch, args.workload, B, rank, local_rank, args, args.steps, args.warmup, flush=flush, barrier=barrier,
                         keep_outputs=bool(args.dump_outputs))
    clocks = sampler.stop()  # sampled across the device-resident and the end-to-end timed regions
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, m.pop("outputs"), prefix=f"rank{rank}_" if world > 1 else "")
    # the one collective of the path: aggregate iterations / residual norm (SUM) and elapsed device time (MAX over ranks)
    from momentum_b200.distributed import aggregate_solve_stats

    its_total, err_total, max_ms = aggregate_solve_stats(float(m["its_per_step"]), m["err_sum"], m["total_ms"], device="cuda")
    value = its_total * args.steps / (max_ms * 1e-3)
    te = torch.tensor([m["e2e_s"]], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = its_total * args.steps / te.item()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    kernels, jtj_phase, kms, st = kernel_report(m, peaks, args.workload)
    dominant = max(kernels, key=lambda k: k["ms_per_launch"])
    line = {
        "metric": "GN iterations/sec (batched 72-joint IK)", "value": value, "unit": "GN it/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": max_ms / args.steps, "higher_is_better": True, "scaling": "strong" if args.strong else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(args, world),
        "solves_per_sec": value / ITERS, "aggregate_final_error": err_total,
        "e2e": {"value": e2e_value, "unit": "GN it/s", "h2d_bytes_per_step": m["h2d"], "d2h_bytes_per_step": m["d2h"], "step_ms": [round(x, 3) for x in m["e2e_step_ms"]]},
        "gpu_launches": int(m["launches"]),
        "clocks": clocks,
        "roofline": dominant,
        "roofline_all_kernels": kernels,
        "jtj": jtj_phase,
        "kernels_ms_per_iteration": kms,
        "path": {0: "three kernels per iteration", 1: "persistent whole-solve kernel", 2: "sweep + gramCholesky per iteration"}[m["fused"]["fused"]],
        "plan": {"tiles": st["cholesky_tiles"], "levels": st["cholesky_levels"], "strip_floats": st["strip_floats"], "gram_pairs": st["gram_pairs"]},
    }
    if world == 1 and not args.no_extras:
        del m
        line["other_workloads"] = extra_workloads(ms, torch, args, rank, local_rank, flush, barrier, peaks)
    if not args.no_cpu_baseline:
        value_cpu, threads, desc, single, _ = time_cpu_arm(args.workload, 10.0)
        line["cpu_baseline"] = {"value": value_cpu, "unit": "GN it/s", "cores": threads, "kind": "port", "sample": desc, "single_thread_value": single}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
