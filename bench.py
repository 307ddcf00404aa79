#!/usr/bin/env python
"""bench.py -- OBCA trajectories/sec on BASELINE config 2 (reverse parking, N=80, 3 obstacles, batch 4096 per GPU).

A "step" = one pass of the hot path over one batch of synthetic problems: DualMultWS (K2) + the batched
interior-point solve (rounds of k_pk_eval [K1] / k_pk_sweep [K3] / k_pk_step [K4], then the persistent tail kernel) of
ParkingSignedDist for B randomised start poses.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU, NCCL); the batch is sharded by rank (weak scaling: B per GPU),
nothing is exchanged on the solve path, one all-reduce carries the counters.  Rank 0 prints ONE JSON line.

--dump-outputs DIR: rank 0 writes what the solver returned in the last timed step as DIR/<name>.npy (float64; see dump_outputs).
The inputs are seeded, so two builds run with the same arguments can be compared output for output.

  value      converged trajectories / s, inputs resident in HBM, device time from CUDA events on the library's
             stream (max over ranks)
  e2e        same metric through the reference-facing C-ABI call with pinned HOST buffers (H2D + D2H inside)
  roofline   dominant kernel (k_pk_eval = K1 of the rounds) against the measured HBM peak, algorithmic bytes of SURVEY 8(d)
  cpu_baseline / --impl reference : the oracle port (IPOPT stand-in, oracle/ipm_ref.py sparse path) on host cores
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

for _v in ("OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):   # numpy's BLAS stays single-threaded; the CPU arms use OpenMP over problems
    os.environ.setdefault(_v, "1")

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_HORIZON = 80
WORKLOAD = "reverse-parking SD var-time, N=80, 3 obstacles vOb=[2,2,1] (BASELINE config 2)"
# SURVEY.md 8(d): fused K1 (J/H never reach HBM): 8*(2n+2m+n_par), n=2185, m=1460, n_par=243
ALG_BYTES_PER_EVAL = 8 * (2 * 2185 + 2 * 1460 + 243)


def ncu_traffic():
    """DRAM bytes (read + write) of one k_pk_eval launch with all 4096 problems active, from the committed ncu capture
    (profiles/ncu_traffic_r02.json, written by tools/ncu_traffic.py from `ncu --set full`), or None."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic_r02.json")
    if not os.path.exists(p):
        return None
    L = json.load(open(p))["launches"]
    ev = [e for e in L if e["kernel"].startswith("k_pk_eval")]
    return (ev[0]["dram_read_bytes"] + ev[0]["dram_write_bytes"]) if ev else None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------------------
# CPU arm: the compiled oracle port on host cores
# ----------------------------------------------------------------------------------------------------------
CPU_KIND = ("port (oracle/cpu_ipm: compiled C++ generic sparse interior point = the published Ipopt algorithm as restated in "
            "oracle/ipm_ref.py, sympy-generated derivatives of the reference-formulation NLP, skyline LDL' of the full augmented "
            "system; IPOPT stand-in, not IPOPT)")


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


class CpuArm:
    """n problems of the benchmark batch (seed 0) prepared once (model build: python, reported, not timed -- the reference's JuMP
    model build is outside its `time` too); run() = DualMultWS (DualMultWS.jl:36-77) + solve(m) (ParkingSignedDist.jl:240) for all
    of them, one problem per OpenMP thread."""

    def __init__(self, n, threads):
        from obca_b200.scenarios import reverse_parking_batch
        from oracle import cpu_ipm
        self.n, self.threads = n, threads
        t0 = time.time()
        cpu_ipm.build()
        self.call = cpu_ipm.ParkingCall(reverse_parking_batch(n, N_HORIZON, 0), range(n), "sd", 0)
        self.setup_s = time.time() - t0

    def run(self):
        r = self.call.run(nthreads=self.threads)
        conv = int((r["status"] == 1).sum())
        return dict(conv=conv, wall=r["wall_dualws"] + r["wall_solve"], wall_solve=r["wall_solve"], wall_dualws=r["wall_dualws"],
                    iters=float(r["iters"].mean()), per_solve=float(r["seconds"].mean()),
                    per_dualws=float(r["dualws"]["seconds"].mean()))


def best_threads(arm, threads):
    """The host may expose more logical CPUs than it can run the solves on at full speed (SMT, memory bandwidth, cgroup quota):
    time the same prepared sample with threads, threads/2, threads/4, threads/8 and keep the best throughput."""
    best = None
    for t in sorted({threads, max(1, threads // 2), max(1, threads // 4), max(1, threads // 8)}, reverse=True):
        arm.threads = t
        a = arm.run()
        if best is None or a["conv"] / a["wall"] > best[1]["conv"] / best[1]["wall"]:
            best = (t, a)
    arm.threads = best[0]
    return best


def cpu_baseline_line(threads):
    """Bounded sample: 4 problems per host thread of the benchmark batch; the best thread count + a single-thread figure."""
    arm = CpuArm(4 * threads, threads)
    arm.run()                                   # warm-up (page-in, OpenMP pool)
    t_best, a = best_threads(arm, threads)
    one = CpuArm(8, 1)
    o = one.run()
    return {"value": a["conv"] / a["wall"], "unit": "traj/s", "cores": t_best, "kind": CPU_KIND,
            "sample": f"{arm.n} problems of the same batch (seed 0), one per OpenMP thread, {t_best} threads (best of {threads} and fractions of it on a "
                      f"{threads}-CPU host), DualMultWS + solve {a['wall']:.2f} s wall (solve alone {a['wall_solve']:.2f} s = the reference's `time` "
                      f"semantic), mean {a['per_solve'] * 1e3:.0f} ms/solve + {a['per_dualws'] * 1e3:.0f} ms DualMultWS, mean {a['iters']:.0f} iterations; "
                      f"model build (python, untimed) {arm.setup_s:.1f} s",
            "solve_only_value": a["conv"] / a["wall_solve"],
            "single_thread_value": o["conv"] / o["wall"], "single_thread_solve_only_value": o["conv"] / o["wall_solve"]}


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_cores()
    arm = CpuArm(args.cpu_sample or 4 * threads, threads)          # one step = 4 problems per host thread (--cpu-sample: tests)
    arm.run()
    threads_used, _ = best_threads(arm, threads)      # (warm-up; all the host threads it can use)
    for _ in range(max(args.warmup - 1, 0)):
        arm.run()
    t0 = time.time(); conv = 0; its = []; solve_s = 0.0
    for _ in range(args.steps):
        a = arm.run()
        conv += a["conv"]; its.append(a["iters"]); solve_s += a["wall_solve"]
    wall = time.time() - t0
    val = conv / wall
    line = {"impl": "reference", "metric": "OBCA trajs/sec, reverse-parking N=80 3-obs batch", "value": val, "unit": "traj/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample_per_step": arm.n, "iters_mean": float(np.mean(its)),
                       "solve_only_traj_per_s": conv / solve_s, "model_build_s_untimed": arm.setup_s},
            "cpu_baseline": {"value": val, "unit": "traj/s", "cores": threads_used, "kind": CPU_KIND,
                             "sample": f"{arm.n} problems/step of the same batch (seed 0), one per OpenMP thread ({threads_used} threads: best of "
                                       f"{threads} and fractions of it), DualMultWS + solve timed; "
                                       "model build untimed (as in the reference's `time`)"},
            "e2e": {"value": val, "unit": "traj/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ----------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, dev):
        super().__init__(daemon=True)
        self.dev = dev; self.stop = False; self.sm = []; self.reasons = set(); self.sm_max = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(dev)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons)}


def gpu_arm(args):
    import torch
    import obca_b200
    from obca_b200 import scenarios
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    from obca_b200 import sharding
    dist = None
    cpus = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        cpus = sharding.pin_rank_to_cpus(local, int(os.environ.get("LOCAL_WORLD_SIZE", world)))   # one CPU slice per rank
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = obca_b200.lib()
    N, NS = N_HORIZON, N_HORIZON + 1
    if args.scaling == "strong":
        # strong scaling: ONE global batch of --batch problems (seed 0), rank r solves its contiguous slice (sharding.shard_batch)
        sc = sharding.shard_batch(scenarios.reverse_parking_batch(args.batch, N, seed=0), world, rank)
    else:
        sc = scenarios.reverse_parking_batch(args.batch, N, seed=rank)      # weak scaling: --batch independent problems per rank
    B = sc["B"]
    nOb, V = sc["nOb"], int(np.sum(sc["vOb"]))
    vOb = np.ascontiguousarray(sc["vOb"], np.int32); A = np.asfortranarray(sc["A"]); b = np.ascontiguousarray(sc["b"]).ravel()
    ego = np.ascontiguousarray(sc["ego"]); xyb = np.ascontiguousarray(sc["XYbounds"])
    host_in = dict(x0=sc["x0"], xF=np.broadcast_to(sc["xF"], (B, 4)), rx=sc["rx"], ry=sc["ry"], ryaw=sc["ryaw"],
                   xWS=np.transpose(sc["xWS"], (0, 2, 1)), uWS=np.transpose(sc["uWS"], (0, 2, 1)))
    hin = {k: torch.from_numpy(np.ascontiguousarray(v, dtype=np.float64)).pin_memory() for k, v in host_in.items()}
    din = {k: v.cuda(non_blocking=True) for k, v in hin.items()}
    shapes = dict(xp=(B, NS, 4), up=(B, N, 2), ts=(B, NS), lp=(B, NS, V), np=(B, NS, 4 * nOb), sl=(B, NS, nOb), err=(B,))
    dout = {k: torch.zeros(s, dtype=torch.float64, device="cuda") for k, s in shapes.items()}
    hout = {k: torch.zeros(s, dtype=torch.float64).pin_memory() for k, s in shapes.items()}
    dflag = torch.zeros(B, dtype=torch.int32, device="cuda"); dit = torch.zeros(B, dtype=torch.int32, device="cuda")
    hflag = torch.zeros(B, dtype=torch.int32).pin_memory(); hit = torch.zeros(B, dtype=torch.int32).pin_memory()
    opts = obca_b200.default_opts(device=local, retry=1)
    sec = np.zeros(1)
    t_ws = C.c_double(0.0); t_sv = C.c_double(0.0); ws_s = [0.0]; sv_s = [0.0]
    P = lambda t: C.c_void_p(t.data_ptr())
    NP = lambda a: a.ctypes.data_as(C.c_void_p)

    def step_dev():
        rc = lib.obca_parking_solve_batch_dev(C.c_int(B), C.c_int(N), C.c_int(nOb), NP(vOb), NP(A), NP(b), P(din["x0"]), P(din["xF"]),
                                              C.c_double(sc["Ts"]), C.c_double(sc["L"]), NP(ego), NP(xyb), P(din["rx"]), P(din["ry"]),
                                              P(din["ryaw"]), P(din["xWS"]), P(din["uWS"]), None, None, C.c_int(0), C.c_int(1),
                                              C.byref(opts), P(dout["xp"]), P(dout["up"]), P(dout["ts"]), P(dout["lp"]), P(dout["np"]),
                                              P(dout["sl"]), P(dflag), P(dit), P(dout["err"]), NP(sec))
        assert rc == 0, lib.obca_last_error()
        # solve_seconds is the reference's `time` (solve only, ParkingSignedDist.jl:239-241); the step of the hot path also
        # contains DualMultWS (:219): both event-timed on the library's stream
        lib.obca_last_times(C.c_int(local), C.byref(t_ws), C.byref(t_sv))
        ws_s[0] += t_ws.value; sv_s[0] += t_sv.value
        return t_ws.value + t_sv.value

    def step_host():
        rc = lib.obca_parking_solve_batch(C.c_int(B), C.c_int(N), C.c_int(nOb), NP(vOb), NP(A), NP(b), P(hin["x0"]), P(hin["xF"]),
                                          C.c_double(sc["Ts"]), C.c_double(sc["L"]), NP(ego), NP(xyb), P(hin["rx"]), P(hin["ry"]),
                                          P(hin["ryaw"]), P(hin["xWS"]), P(hin["uWS"]), None, None, C.c_int(0), C.c_int(1),
                                          C.byref(opts), P(hout["xp"]), P(hout["up"]), P(hout["ts"]), P(hout["lp"]), P(hout["np"]),
                                          P(hout["sl"]), P(hflag), P(hit), P(hout["err"]), NP(sec))
        assert rc == 0, lib.obca_last_error()

    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device="cuda")   # > 126 MB L2
    torch.cuda.synchronize()      # the library runs on its own stream: the torch-side copies / fills above must have landed

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_dev()
    step_host()
    # ---- device-resident timing ----
    sampler = ClockSampler(local); sampler.start()
    barrier()
    t_wall0 = time.perf_counter()
    dev_s = 0.0; ws_s[0] = 0.0; sv_s[0] = 0.0
    for _ in range(args.steps):
        flush.zero_(); torch.cuda.synchronize()
        dev_s += step_dev()
    barrier()
    wall_s = time.perf_counter() - t_wall0
    if args.dump_outputs and rank == 0:      # before the e2e and profiling solves below reuse the device buffers
        dump_outputs(args.dump_outputs, dict(xp=dout["xp"], up=dout["up"], ts=dout["ts"], lp=dout["lp"], np=dout["np"], sl=dout["sl"],
                                             exitflag=dflag, iters=dit, kkt_err=dout["err"]))
    conv = int(dflag.sum().item()); it_sum = int(dit.sum().item()); it_max = int(dit.max().item())
    evals = it_sum + B
    # ---- end-to-end through the host-pointer C-ABI ----
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host()
    barrier()
    e2e_s = time.perf_counter() - t0
    sampler.stop = True; sampler.join()
    conv_h = int(hflag.sum().item())
    # the collectives of the path (obca_b200.sharding): counters SUM over NVLink, times MAX over the ranks
    red = sharding.reduce_stats(dist, "cuda", dict(conv=conv, conv_h=conv_h, it_sum=it_sum, evals=evals, problems=B),
                                dict(dev_s=dev_s, e2e_s=e2e_s, wall_s=wall_s))
    dev_s, e2e_s, wall_s = red["dev_s"], red["e2e_s"], red["wall_s"]
    conv_all, conv_h_all, it_all, evals_all, B_all = red["conv"], red["conv_h"], red["it_sum"], red["evals"], red["problems"]
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    hbm, how = peaks()
    value = conv_all / (dev_s / args.steps)
    e2e_val = conv_h_all / (e2e_s / args.steps)
    kernel_s = dev_s / args.steps                        # the solver kernels are (all but the K2 launch) the event-bracketed step
    achieved = (evals_all / world) * ALG_BYTES_PER_EVAL / kernel_s / 1e9
    h2d = sum(int(v.numel()) * 8 for v in hin.values())
    d2h = sum(int(v.numel()) * 8 for v in hout.values()) + 8 * B
    line = {"metric": "OBCA trajs/sec, reverse-parking N=80 3-obs batch", "value": value, "unit": "traj/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dev_s / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": B, "global_batch": int(B_all), "parallelism": f"batch-shard x{world}",
                       "cpu_pinning_rank0": (f"{len(cpus)} CPUs" if cpus else "none"),
                       "l2": "256 MB flush between timed steps", "tol": 1e-5, "max_iter": 200,
                       "converged_frac": conv_all / B_all, "iters_mean": it_all / B_all, "iters_max_rank0": it_max,
                       "wall_ms_per_step": 1e3 * wall_s / args.steps,
                       "dualws_ms_per_step_rank0": 1e3 * ws_s[0] / args.steps,
                       "solve_only_ms_per_step_rank0": 1e3 * sv_s[0] / args.steps},
            "clocks": sampler.result(),
            "e2e": {"value": e2e_val, "unit": "traj/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": 2 * args.steps,
            "roofline": {"bound": "hbm", "kernel": "whole solve: rounds of k_pk_eval/k_pk_sweep/k_pk_step<2,true>, then k_pk_tail<2,true>", "achieved": achieved, "peak": hbm, "unit": "GB/s",
                         "frac": achieved / hbm, "traffic": None,
                         "note": f"algorithmic bytes = {ALG_BYTES_PER_EVAL} B x (iterations+1) per problem (SURVEY 8d, fused K1); "
                                 f"peak {how}; the solver is FP64-latency bound, see DESIGN.md and profiles/"}}
    # ---- acceptance of the end-to-end outputs by the reference's own checker (k_check through the C-ABI) + iteration histogram ----
    try:
        from obca_b200 import parking as _pk
        T_ = lambda t: np.transpose(t.numpy(), (0, 2, 1))
        feas, _, strict = _pk.check_parking_batch(sc["x0"], sc["xF"], N, sc["Ts"], sc["L"], sc["ego"], sc["XYbounds"], nOb, sc["vOb"], sc["A"],
                                                  sc["b"], T_(hout["xp"]), T_(hout["up"]), T_(hout["lp"]), T_(hout["np"]), hout["ts"].numpy(), 0, 1,
                                                  T_(hout["sl"]), opts)
        line["config"]["checker_pass_frac_rank0"] = float(np.mean(feas))        # verbatim ParkingConstraints (5e-5)
        line["config"]["strict_audit_pass_frac_rank0"] = float(np.mean(strict))
        line["config"]["iters_hist_by_10_rank0"] = np.bincount(np.minimum(hit.numpy() // 10, 20), minlength=21).tolist()
    except Exception as e:                                                       # diagnostic only: never fail the bench line
        line["config"]["checker_pass_frac_rank0"] = None
        line["config"]["checker_note"] = repr(e)[:160]
    # ---- K1 stand-alone (fused constraint / Lagrangian-gradient evaluation) at the solution points: HBM roofline ----
    nn = C.c_longlong(); mm = C.c_longlong()
    lib.obca_parking_eval_sizes(C.c_int(N), C.c_int(nOb), NP(vOb), C.c_int(1), C.byref(nn), C.byref(mm))
    n_z, m_c = nn.value, mm.value
    yk1 = torch.randn((B, m_c), dtype=torch.float64, device="cuda")
    ck1 = torch.empty((B, m_c), dtype=torch.float64, device="cuda"); gk1 = torch.empty((B, n_z), dtype=torch.float64, device="cuda")
    fk1 = torch.empty((B, NS), dtype=torch.float64, device="cuda")
    k1ms = np.zeros(1)

    def k1(reps):
        rc = lib.obca_parking_eval_batch_dev(C.c_int(B), C.c_int(N), C.c_int(nOb), NP(vOb), NP(A), NP(b), P(din["x0"]), P(din["xF"]),
                                             C.c_double(sc["Ts"]), C.c_double(sc["L"]), NP(ego), NP(xyb), P(din["rx"]), P(din["ry"]),
                                             P(din["ryaw"]), P(dout["xp"]), P(dout["up"]), P(dout["ts"]), P(dout["lp"]), P(dout["np"]),
                                             P(dout["sl"]), P(yk1), C.c_int(0), C.c_int(1), C.byref(opts), P(ck1), P(gk1), P(fk1),
                                             C.c_int(reps), NP(k1ms))
        assert rc == 0, lib.obca_last_error()
        return float(k1ms[0])
    k1(3)
    k1_ms = k1(20)
    k1_bytes = 8.0 * (2 * n_z + 2 * m_c + 3 * NS) * B
    k1_gbs = k1_bytes / (k1_ms * 1e-3) / 1e9
    line["roofline_k1"] = {"bound": "hbm", "kernel": "k_parking_eval<2,true>", "achieved": k1_gbs, "peak": hbm, "unit": "GB/s",
                           "frac": k1_gbs / hbm, "traffic": None, "ms_per_launch": k1_ms,
                           "note": f"stand-alone fused K1: 8*(2n+2m+3(N+1)) = {int(k1_bytes / B)} B/problem/evaluation, B={B}; working set "
                                   f"{k1_bytes / 1e6:.0f} MB > L2; mean of 20 back-to-back launches"}
    rnd = C.c_int(0); hand = C.c_int(0); kms = (C.c_double * 5)()
    if lib.obca_last_schedule(C.c_int(local), C.byref(rnd), C.byref(hand), None) == 0:
        line["config"]["schedule"] = {"phase_split_rounds": rnd.value, "handed_to_tail_kernel": hand.value}
        # launches of our kernels per step: DualMultWS + 3 per round + the tail kernel; device arm + e2e arm
        line["gpu_launches"] = args.steps * (1 + 3 * rnd.value + (1 if hand.value > 0 else 0)) * 2
        # one extra, untimed solve with CUDA events around every kernel: which kernel dominates the step, and the live K1 roofline
        os.environ["OBCA_PHASE_TIMING"] = "1"
        step_dev()
        os.environ.pop("OBCA_PHASE_TIMING", None)
        pr = (C.c_ulonglong * 8)()
        if lib.obca_last_schedule(C.c_int(local), C.byref(rnd), None, kms) == 0 and lib.obca_last_profile(C.c_int(local), pr) == 0:
            names = ["k_pk_eval (K1: constraint blocks + stage terms + assembly + decisions)", "k_pk_sweep (K3 KKT)",
                     "k_pk_step (K4 recovery, line search, update)", "k_pk_tail (persistent, all phases)", "k_dualws (K2)"]
            tot = sum(kms) or 1.0
            line["kernel_share"] = {n: round(kms[i] / tot, 4) for i, n in enumerate(names)}
            line["kernel_ms_event_timed"] = {n: round(kms[i], 3) for i, n in enumerate(names)}
            ev_r, ev_r2, me_r, ev_t, me_t = int(pr[7]), int(pr[5]), int(pr[6]), int(pr[4]), int(pr[3])
            line["phase_counts"] = {"k1_evals_rounds": ev_r, "of_which_after_barrier_update": ev_r2, "merit_evals_rounds": me_r,
                                    "k1_evals_tail": ev_t, "merit_evals_tail": me_t}
            if ev_r > 0 and kms[0] > 0 and rnd.value > 0:
                # K1 = k_pk_eval: the largest kernel of the step.  Algorithmic bytes: SURVEY 8d, fused variant (J/H never reach HBM
                # as matrices), 60 264 B per problem per evaluation, times the evaluations the kernel did (device counter).
                t_k1 = kms[0] * 1e-3
                ach = ev_r * ALG_BYTES_PER_EVAL / t_k1 / 1e9
                line["roofline_solve"] = line["roofline"]
                line["roofline"] = {"bound": "hbm", "kernel": "k_pk_eval<2,true> (K1 of the rounds)", "achieved": ach,
                                    "peak": hbm, "unit": "GB/s", "frac": ach / hbm, "traffic": ncu_traffic(),
                                    "launches": rnd.value, "ms_per_launch": 1e3 * t_k1 / rnd.value, "evaluations": ev_r,
                                    "note": f"achieved = {ALG_BYTES_PER_EVAL} B (SURVEY 8d, fused K1) x {ev_r} K1 evaluations of one solve (device counter) / "
                                            f"summed CUDA-event time of the {rnd.value} k_pk_eval launches on the library's stream; peak {how}; traffic = dram "
                                            "read + write of ONE launch with all 4096 problems active (ncu --set full, profiles/ncu_traffic_r02.json): iterate "
                                            "in, stage slots (53 KB) + local maps (47 KB) + iterate state out; the block hand-over stays in shared memory"}
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline_line(host_cores())
        # second CPU figure: the SAME structure-exploiting algorithm as the kernels (block condensation + Riccati sweep), i.e. the
        # per-stage CUDA source compiled by g++ for the host (tests/emul, test infrastructure: the emulation the CPU tests check
        # the kernels' arithmetic with), one problem per OpenMP thread.  What a CPU gets out of this solver design; not IPOPT.
        try:
            sys.path.insert(0, os.path.join(ROOT, "tests", "emul"))
            import emul
            nprob = min(1024, 8 * host_cores())
            scc = scenarios.reverse_parking_batch(nprob, N, seed=0)
            try:      # the emulation's `omp parallel for` takes the global thread count (torch / the launcher may have set it to 1)
                C.CDLL("libgomp.so.1").omp_set_num_threads(C.c_int(host_cores()))
            except OSError:
                pass
            emul.lib()
            t0 = time.time()
            lpe, npe, _, _ = emul.dualmultws_batch(scc)
            re_ = emul.solve_batch(scc, 0, "sd", None, lpe, npe)
            wall_e = time.time() - t0
            line["cpu_structured"] = {"value": float((re_["status"] == 1).sum()) / wall_e, "unit": "traj/s", "cores": host_cores(),
                                      "kind": "port (host build of the kernels' own per-stage source, OpenMP over problems)",
                                      "sample": f"{nprob} problems of the same batch (seed 0), {wall_e:.1f} s wall, DualMultWS + solve"}
        except Exception as e:      # the emulation is optional test infrastructure
            line["cpu_structured"] = {"unavailable": repr(e)[:200]}
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


def gpu_arm_other(args):
    """The other BASELINE configurations (not the headline line): --workload parallel | parallel4 | quadcopter | dist |
    fixed.  Same timing rules; goes through the reference-facing host API (obca_b200.parking / .quadcopter), so `value`
    is the device-timed solve (CUDA events inside the library, inputs resident) and `e2e` the wall clock of the call
    with host buffers."""
    import torch
    import obca_b200
    from obca_b200 import parking, quadcopter, scenarios
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    w = args.workload
    B = args.batch
    opts = obca_b200.default_opts(device=local, retry=1)
    if w == "quadcopter":
        B = min(B, 2048) if args.batch == 4096 else B
        sc = scenarios.quadcopter_batch(B, 100, seed=2 + rank)
        name = "QuadcopterSignedDist 3D nav, N=100, 5 box obstacles, 12 states (BASELINE config 4)"
        opts.max_iter = 3000       # the reference sets no max_iter for this model (QuadcopterSignedDist.jl:28-31): Ipopt default
        run = lambda: quadcopter.quadcopter_solve_batch(sc["x0"], sc["xF"], sc["N"], sc["Ts"], sc["R"], sc["obs"], sc["xWS"], 1.0, 1, opts)
        ok = lambda r: int((r["exitflag"] >= 1).sum())
    else:
        fix, sd = (1 if w == "fixed" else 0), (0 if w == "dist" else 1)
        if w in ("parallel", "parallel4"):
            sc = scenarios.parallel_parking_batch(B, N_HORIZON, seed=1 + rank, n_obstacles=4 if w == "parallel4" else 3)
            name = f"parallel-parking SD var-time, N=80, {sc['nOb']} obstacles (BASELINE config 3)"
        else:
            sc = scenarios.reverse_parking_batch(B, N_HORIZON, seed=rank)
            name = f"reverse-parking {'SD' if sd else 'Dist'} {'fixed' if fix else 'var'}-time, N=80, 3 obstacles"
        Ts = sc["Ts_fix"] if fix else sc["Ts"]
        run = lambda: parking.parking_solve_batch(sc["x0"], sc["xF"], sc["N"], Ts, sc["L"], sc["ego"], sc["XYbounds"], sc["nOb"], sc["vOb"],
                                                  sc["A"], sc["b"], sc["rx"], sc["ry"], sc["ryaw"], fix, sc["xWS"], sc["uWS"], sd, None, None, opts)
        ok = lambda r: int(r["exitflag"].sum())
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device="cuda")

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(args.warmup):
        r = run()
    sampler = ClockSampler(local); sampler.start()
    barrier()
    dev_s = 0.0; e2e_s = 0.0; conv = 0; its = 0
    for _ in range(args.steps):
        flush.zero_(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = run()
        e2e_s += time.perf_counter() - t0
        dev_s += r["time"]; conv += ok(r); its += int(r["iters"].sum())
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {k: v for k, v in r.items() if k != "time"})
    sampler.stop = True; sampler.join()
    stats = torch.tensor([dev_s, e2e_s], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([conv, its], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX); dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    dev_s, e2e_s = [float(x) for x in stats.tolist()]
    conv_all, its_all = [float(x) for x in cnt.tolist()]
    if rank == 0:
        line = {"metric": "OBCA trajs/sec (other BASELINE configuration)", "value": conv_all / dev_s, "unit": "traj/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dev_s / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": name, "batch_per_gpu": B, "global_batch": B * world, "parallelism": f"batch-shard x{world}",
                           "l2": "256 MB flush between timed steps", "converged_frac": conv_all / (B * world * args.steps),
                           "iters_mean": its_all / (B * world * args.steps)},
                "clocks": sampler.result(),
                "e2e": {"value": conv_all / e2e_s, "unit": "traj/s", "note": "wall clock of the host-pointer call (H2D + solve + D2H)"}}
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


DUMP_BYTES = 64 * 10**6


def dump_outputs(out_dir, arrays):
    """Writes one step's outputs (arrays or tensors with the problem index on axis 0) as out_dir/<name>.npy in float64.  When all
    of them would exceed DUMP_BYTES, a sample of the problems drawn with a fixed seed is written instead, the same for every run
    with the same batch; problem.npy holds the batch indices of the rows written (all of them when nothing was dropped)."""
    arrays = {k: np.asarray(v.cpu() if hasattr(v, "cpu") else v, dtype=np.float64) for k, v in arrays.items()}
    B = len(next(iter(arrays.values())))
    per_problem = 8 * (1 + sum(a[0].size for a in arrays.values()))
    n = min(B, (DUMP_BYTES - 1024 * (len(arrays) + 1)) // per_problem)          # 1 KB per file for the .npy header
    idx = np.arange(B) if n == B else np.sort(np.random.default_rng(0).choice(B, n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "problem.npy"), idx.astype(np.float64))
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a[idx])


_OUT_FD = None


def emit(line):
    """The ONE JSON line of the run, on the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _OUT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_OUT_FD, data)


def main():
    # stdout carries exactly one JSON line: whatever libraries print on file descriptor 1 during the run (NCCL's version banner at
    # NCCL_DEBUG=VERSION / WARN / INFO, for one) is sent to stderr; emit() writes the line to the original stdout.
    global _OUT_FD
    sys.stdout.flush()
    _OUT_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--impl", default="obca")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=0, help="problems per step of the CPU arm (default: 4 per host thread)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (default, the headline): --batch problems PER GPU; strong: --batch problems in total, sharded over the GPUs")
    ap.add_argument("--workload", default="reverse", choices=["reverse", "parallel", "parallel4", "quadcopter", "dist", "fixed"],
                    help="reverse = BASELINE config 2 (the headline line, default); the others print a secondary line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the solver outputs of the last timed step to DIR/<name>.npy (GPU arms; at most 64 MB, sampled by problem above that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arms; the reference arm returns none")
    if args.impl == "reference":
        reference_arm(args)
    elif args.workload != "reverse":
        gpu_arm_other(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
