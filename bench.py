#!/usr/bin/env python
"""bench.py -- EI candidates/sec of the GP-EI chooser hot path, and chooser.next() wall-ms (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME]

A "step" is one pass of ``ei_over_hypers`` (chooser/GPEIOptChooser.py:331-341 of the reference) over the
whole candidate grid for all S hyper-samples: K build -> Cholesky -> explicit inverse + alpha -> cross-covariance
generator -> tcgen05 predict GEMM (3xFP16 scaled split) -> EI sweep (-> all-reduce of the per-candidate EI sum when
N > 1) -> argmax.

  value : M / step-time with X, candidates, values and hyper-samples already resident in HBM.
  e2e   : the same metric through the reference-facing plugin call (``chooser.ei_over_hypers(comp, pend, cand, vals)``:
          host numpy in, (M, S) float64 EI matrix out, then the host argmax of the mean), host<->device copies inside
          the timed region, --steps iterations.
  roofline     : the dominant kernel (tc::predict_tc_kernel, the N^2*M triangular-solve term as a GEMM against the
                 explicit inverse): algorithmic flops / its CUDA-event time vs the measured dense bf16 tensor peak
                 (MEASURED_PEAKS.json); traffic = DRAM bytes per launch read from the committed ncu summary
                 profiles/r02_predict_tc_traffic.json (bench.py never runs under a profiler).
  cpu_baseline : the oracle port (oracle.gp_oracle.compute_ei: the reference's own numpy/scipy operation sequence,
                 GPEIOptChooser.py:527-556) timed on this box's host cores -- BLAS threads pinned to all of them, the same
                 at every --gpus N -- on a bounded sample and extrapolated linearly (the reference loop is exactly
                 linear in S and, for fixed N, affine in M).  Its EI values are compared with the GPU's
                 (``parity``: max |dEI| / max EI over the sample, argmax equality).
  next  : chooser.next() wall-ms through the plugin API at the SAME workload, steady state (no burn-in), with the phase
          split (MCMC / grid pass 1 / L-BFGS refinement / grid pass 2) and the CPU port's time as counts x unit times.
  --impl reference : the CPU implementation as its own arm (rank 0 only).
  --dump-outputs DIR : after the timed steps, what the last step of each EI leg returned: ei_sum (M,) and argmax of the
          value leg, ei_matrix_e2e (M, S) and argmax_e2e of the e2e leg.  The inputs are seeded, so two builds run with
          the same arguments can be compared output for output.

Multi-GPU: hyper-samples are sharded round-robin over ranks (total work fixed -> "scaling": "strong"); the
only exchange is one NCCL all-reduce of M floats.
"""
import os
import sys

# BLAS / OpenMP threads of the CPU arm: all host cores, decided HERE, before numpy loads its BLAS.  torchrun exports
# OMP_NUM_THREADS=1 to every rank; without this the CPU baseline would be ~2.4x slower under --gpus N > 1 than at N = 1.
_CORES = os.cpu_count() or 1
for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ[_v] = str(_CORES)

import argparse   # noqa: E402
import ctypes     # noqa: E402
import json       # noqa: E402
import subprocess  # noqa: E402
import tempfile   # noqa: E402
import threading  # noqa: E402
import time       # noqa: E402

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (D, N, M, S)           BASELINE.json configs / metric
    "headline": (32, 4096, 100000, 40),   # "EI candidates/sec (N=4096 obs, 100k cands, 40 hypers)"
    "c2": (8, 512, 10000, 10),
    "c3": (20, 2048, 50000, 20),
    "c4": (8, 1024, 20000, 10),           # GPEIperSecChooser dual GP (objective + cost); D, S: SURVEY 8 defaults
    "c5": (32, 8192, 100000, 40),
    "tiny": (4, 96, 2000, 4),
}
PER_SECOND = ("c4",)                       # workloads that run the EI-per-second path (PSEC:437-548)
KIND = "Matern52"


def synth(D, N, M, S):
    """SURVEY.md 8(d) synthetic problem; the grid is RandomState(0).rand (not Sobol: generation time only)."""
    grid = np.random.RandomState(0).rand(N + M, D)
    perm = np.random.RandomState(0).permutation(N + M)
    complete, candidates = np.sort(perm[:N]), np.sort(perm[N:])
    comp, cand = grid[complete], grid[candidates]
    y = np.sin(3 * comp).sum(1) + 0.01 * np.random.RandomState(1).randn(N)
    vals = (y - y.mean()) / y.std()
    rs = np.random.RandomState(2)
    hs = [(0.1 * rs.randn(), 1e-3, float(np.exp(0.25 * rs.randn())), rs.uniform(0.3, 2.0, D)) for _ in range(S)]
    return comp, cand, vals, hs


def synth_time(D, comp, S):
    """Duration GP of the per-second workloads: durations = 1 + x_0 (SURVEY 8d), its own hyper-samples."""
    durs = np.log(1.0 + comp[:, 0])
    rs = np.random.RandomState(5)
    ths = [(float(np.mean(durs)) + 0.05 * rs.randn(), 1e-3, float(np.exp(0.25 * rs.randn())), rs.uniform(0.3, 2.0, D))
           for _ in range(S)]
    return durs, ths


def flops_per_pair(N, D):
    """SURVEY.md 8(d): algorithmic flops per (candidate, hyper-sample) pair."""
    return float(N) * N + 2.0 * N * D + 4.0 * N + 25.0 * N + 40.0


def ncu_traffic(workload, impl, world, launches_per_step):
    """DRAM bytes per launch of the dominant kernel from the committed ncu summary (which names its capture commit)."""
    p = os.path.join(ROOT, "profiles", "r02_predict_tc_traffic.json")
    if impl != "tc" or world != 1 or not os.path.exists(p):
        return None, None
    d = json.load(open(p))
    w = d.get("workloads", {}).get(workload)
    if not w:
        return None, None
    return float(w["dram_bytes_per_step"]) / max(1, launches_per_step), "profiles/r02_predict_tc_traffic.json @ %s" % d.get("commit")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tensor_burst=d["bf16_tflops"], tensor_sustained=d["bf16_tflops_sustained"],
                    src="MEASURED_PEAKS.json")
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor_sustained=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler(object):
    """nvidia-smi clock / throttle-reason samples during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc, self.t_begin = index, [], None, 0.0

    def mark_begin(self):
        """Samples from here on count.  The process is started BEFORE the warm-up: nvidia-smi's start-up (driver / NVML
        initialisation over all GPUs of the node) holds driver locks for tens of milliseconds, which showed up as 30-40 ms per
        step in a 3-step timed region when it was started together with it."""
        self.t_begin = time.perf_counter()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t_row, r in self.rows:
            if t_row < self.t_begin:
                continue
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                pw.append(float(r[3]))
                for k, n in enumerate(names):
                    if r[5 + k].lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(np.max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_median": float(np.median(pw)) if pw else None}


# --------------------------------------------------------------------------------------------- CPU arm
def blas_threads():
    """Pins every BLAS / OpenMP pool numpy and scipy loaded to all host cores; returns what is in effect."""
    try:
        import threadpoolctl
        threadpoolctl.threadpool_limits(limits=_CORES)
        info = threadpoolctl.threadpool_info()
        return max([int(i.get("num_threads", 1)) for i in info] or [1])
    except Exception:
        return _CORES


def cpu_port_sample(workload, D, N, M, S, budget_cands=None):
    """Times the oracle port (O.compute_ei / O.compute_ei_per_s: the reference's operation sequence) on host cores on a
    bounded sample and extrapolates to the full (M, S) pass.

    compute_ei is affine in the number of candidates for fixed N (K build + Cholesky + alpha once, then per-candidate
    work) and ei_over_hypers is a plain loop over S (OPT:333-340), so two timings of ONE hyper-sample at m0 and Mc
    candidates give   t_full = S * (t_fixed + t_cand_per * M)."""
    from oracle import gp_oracle as O
    threads = blas_threads()
    comp, cand, vals, hs = synth(D, N, M, S)
    pend = np.zeros((0, D))
    per_s = workload in PER_SECOND
    if per_s:
        durs, ths = synth_time(D, comp, S)

    def one(mc):
        t0 = time.perf_counter()
        if per_s:
            e = O.compute_ei_per_s(KIND, hs[0], ths[0], comp, pend, cand[:mc], vals, durs)
        else:
            e = O.compute_ei(KIND, hs[0], comp, pend, cand[:mc], vals)
        return time.perf_counter() - t0, e

    m0 = min(M, 16)
    one(m0)                                                   # warm-up (BLAS thread pools, page faults)
    t_small, _ = one(m0)
    auto = budget_cands is None
    Mc = int(min(M, budget_cands if not auto else max(500, 2.0e11 / (float(N) * N + 60.0 * N * D))))
    t_big, ei = one(Mc)
    if auto and t_big < 8.0 and Mc < M:                       # many-core hosts: grow the sample to ~15 s of CPU work
        Mc = int(min(M, 60000, max(Mc, Mc * 15.0 / max(t_big - t_small, 1e-3))))   # (<= 2 GB per N x Mc float64 temporary)
        t_big, ei = one(Mc)
    per_cand = max(t_big - t_small, 1e-9) / max(Mc - m0, 1)
    t_fixed = max(t_small - per_cand * m0, 0.0)
    t_full = S * (t_fixed + per_cand * M)
    return dict(value=M / t_full, t_full_s=t_full, t_fixed_s=t_fixed, t_cand_s=per_cand * Mc, Mc=Mc, ei=ei, threads=threads,
                sample="oracle.gp_oracle.%s on 1 of %d hyper-samples, N=%d, %d and %d of %d candidates (%.1f s of CPU "
                       "work, %d BLAS threads); affine fit extrapolated to S=%d, M=%d (t_fixed=%.2fs K+chol+alpha, "
                       "%.3f ms per candidate)" % ("compute_ei_per_s" if per_s else "compute_ei", S, N, m0, Mc, M,
                                                   2 * t_small + t_big, threads, S, M, t_fixed, 1e3 * per_cand))


def run_reference_arm(args, D, N, M, S):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    for it in range(args.warmup + args.steps):
        r = cpu_port_sample(args.workload, D, N, M, S, budget_cands=args.cpu_cands)
        if it >= args.warmup:
            vals.append(r)
    t = float(np.mean([r["t_full_s"] for r in vals]))
    value = M / t
    out = {"impl": "reference", "metric": "EI candidates/sec", "value": value, "unit": "candidates/s",
           "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": "%s D=%d N=%d M=%d S=%d %s" % (args.workload, D, N, M, S, KIND),
                      "note": "oracle port of the reference numpy/scipy path (the py2 reference cannot travel); "
                              "each step times a bounded sample and extrapolates linearly"},
           "cpu_baseline": {"value": value, "unit": "candidates/s", "cores": vals[-1]["threads"], "kind": "port",
                            "sample": vals[-1]["sample"]},
           "e2e": {"value": value, "unit": "candidates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


# --------------------------------------------------------------------------------------------- GPU arm
def run_b200_arm(args, D, N, M, S):
    import torch
    import torch.distributed as dist
    from spearmint_b200 import _lib, parallel
    from spearmint_b200.backend import DeviceBackend

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: the product arm needs a CUDA device (B200, sm_100a) -- there is no CPU fallback; "
                         "the CPU arm is `--impl reference`")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda:%d" % local))
        # The all-cores thread setting at the top of this file is for the CPU arm (rank 0 alone).  Here every rank runs host
        # code of its own (dtype conversions of the uploads are OpenMP loops in torch): N ranks x all cores oversubscribes the
        # host N times.  The plugin call measured 148 ms at 2 GPUs and 139 ms at 8 against 128 / 34 ms of device time -- growing
        # with the rank count, which is what spinning OpenMP teams on an oversubscribed host look like (not re-measured at 8
        # GPUs after this change: the round's GPU budget was spent).  Each rank gets its share of the cores.
        share = max(1, _CORES // world)
        torch.set_num_threads(share)
        try:
            import threadpoolctl
            threadpoolctl.threadpool_limits(limits=share)
        except Exception:
            pass
    backend = DeviceBackend(device="cuda:%d" % local)
    eng = backend.eng32
    comp, cand, vals, hs = synth(D, N, M, S)
    pend = np.zeros((0, D))
    per_s = args.workload in PER_SECOND
    durs, ths = synth_time(D, comp, S) if per_s else (None, None)
    mine = parallel.shard(S, rank, world)
    hs_local = [hs[s] for s in mine]
    ths_local = [ths[s] for s in mine] if per_s else None
    Sl = len(hs_local)

    # ---- resident inputs for the `value` leg
    res = dict(X=eng.to_dev(comp), C=eng.to_dev(cand), y=eng.to_dev(vals), best=float(vals.min()),
               hb=eng.hypers(hs_local, KIND) if Sl else None)
    ldm = ((M + 127) // 128) * 128

    def step_resident():
        if Sl:
            # compute reads the resident tensors; the host arrays ride along only for the accuracy guard's float64
            # re-evaluation of flagged hyper-samples (none at the headline)
            # the positive-definiteness status of the factorisations is read back once, after the timed loop
            # (eng.check_deferred below): a step then ends without a host synchronisation and the next one queues behind it
            _, ei_sum, _ = eng.ei_over_hypers_device(KIND, hs_local, comp, None, cand, vals, want_matrix=False,
                                                     inputs_on_device=res, time_hyper_samples=ths_local, durs_log=durs,
                                                     defer_pd_check=True)
        else:
            ei_sum = torch.zeros((ldm,), dtype=torch.float64, device=eng.device)
        parallel.allreduce_sum_(ei_sum)
        idx, _ = eng.topk(ei_sum, M, 1)
        return ei_sum, idx

    # ---- e2e leg: the plugin call.  GPEIOptChooserB200.ei_over_hypers is the drop-in for OPT:331-341; the per-second
    # plugin's method reproduces the reference's column-0-only early return (PSEC:302), so that workload goes through the
    # backend calls the plugin makes (grid_state + ei_matrix) with every column.
    from spearmint_b200.chooser import GPEIOptChooserB200 as plugin
    ch = plugin.init(tempfile.mkdtemp(), "mcmc_iters=%d,burnin=0,noiseless=1" % S)
    ch._backend = backend
    ch.D, ch.hyper_samples = D, list(hs)

    def step_e2e():
        if per_s:
            st = backend.grid_state(KIND, hs, comp, pend, vals, None, ths, durs)
            ei = backend.ei_matrix(st, cand)
        else:
            ei = ch.ei_over_hypers(comp, pend, cand, vals)        # (M, S) float64 on the host
        return ei, int(np.argmax(ei.mean(axis=1)))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    L = _lib.lib()

    def timed(fn, steps, with_timers=False):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        eng.timers = {} if with_timers else None
        L.smk_timing_enable(1 if with_timers else 0)
        l0 = L.smk_launch_count()
        w0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        wall = time.perf_counter() - w0
        ms = e0.elapsed_time(e1)
        launches = L.smk_launch_count() - l0
        stages = eng.stage_ms()
        eng.timers = None
        t = torch.tensor([ms, wall * 1e3, float(launches)], dtype=torch.float64, device=eng.device)
        if world > 1:
            tmax = t.clone()
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            tsum = t.clone()
            dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
            ms, wall_ms, launches = float(tmax[0]), float(tmax[1]), int(tsum[2])
        else:
            wall_ms = wall * 1e3
        return ms, wall_ms, launches, stages, out

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step_resident()
    eng.check_deferred()
    sampler.mark_begin()
    ms, _, launches, stages, (ei_sum, idx) = timed(step_resident, args.steps, with_timers=True)
    eng.check_deferred()
    if args.dump_outputs and rank == 0:       # copied now: the e2e leg below may reuse the engine's buffers
        dump = {"ei_sum": ei_sum[:M].double().cpu().numpy(), "argmax": np.array([float(idx.cpu()[0])])}
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = ms / args.steps
    value = M / (ms_per_step * 1e-3)

    # kernel spans of the resident leg are read below; freeze them before the e2e leg runs
    span = {}
    for nm in ("predict_tc_kernel", "predict_kernel", "kxt_kernel", "trtri_kernel", "linv_pack_f16"):
        c2 = ctypes.c_int(0)
        span[nm] = (L.smk_timing_ms(nm.encode(), ctypes.byref(c2)), c2.value)

    # ---- e2e leg (host buffers through the plugin call); wall-clock over host + device work, max over ranks
    step_e2e()
    _, wall_ms, _, _, (ei_host, best_idx) = timed(step_e2e, args.steps)
    e2e_ms = wall_ms / args.steps
    if args.dump_outputs and rank == 0:
        dump.update(ei_matrix_e2e=ei_host, argmax_e2e=np.array([float(best_idx)]))
        dump_outputs(args.dump_outputs, dump)
    esz = 4
    n_gp = 2 if per_s else 1
    h2d = esz * (comp.size + cand.size + n_gp * vals.size) + esz * n_gp * Sl * (D + 3)
    d2h = 8 * ldm * (S if world > 1 else Sl)      # the EI matrix is float64 (tail values)

    if rank == 0:
        pk = peaks()
        pairs_local = float(M) * Sl
        impl = eng.predict_impl
        kname = "predict_tc_kernel" if impl == "tc" else "predict_kernel"
        kms_total, cnt_v = span[kname]
        kms_step = kms_total / args.steps                       # all launches of the dominant kernel in one step
        n_launch_step = max(1, cnt_v // args.steps)
        # algorithmic flops handled by that kernel per step (SURVEY 8d): the N^2 triangular-solve term for the tcgen05
        # kernel (the cross-covariance is a separate kernel there), the whole per-pair count for the fused SIMT kernel
        alg = (float(N) * N if impl == "tc" else flops_per_pair(N, D)) * pairs_local
        achieved = alg / (kms_step * 1e-3) / 1e12 if kms_step > 0 else None
        other = {}
        for nm in ("kxt_kernel", "trtri_kernel", "linv_pack_f16"):
            if span[nm][1]:
                other[nm + "_ms_per_step"] = span[nm][0] / args.steps
        traffic, traffic_src = ncu_traffic(args.workload, impl, world, n_launch_step)
        roof = {"kernel": "smk::tc::predict_tc_kernel (tcgen05.mma kind::f16, 3xFP16 scaled split, fp32 accumulate)" if impl == "tc"
                else "smk::predict_kernel<float> (SIMT FMA)",
                "bound": "tensor", "achieved": achieved, "peak": pk["tensor_sustained"], "unit": "TFLOP/s",
                "frac": (achieved / pk["tensor_sustained"]) if achieved else None,
                "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": pk["src"] + " bf16 dense, sustained (kernel timed inside a long step)",
                "algorithmic_flops_per_launch": alg / n_launch_step, "launches_per_step": n_launch_step,
                "kernel_ms_per_launch": kms_step / n_launch_step, "kernel_ms_per_step": kms_step,
                "note": "fp32-accurate results need 3 fp16 MMAs per product (hi*hi + hi*lo + lo*hi, operands scaled by exact "
                        "powers of two): 3 bf16-equivalent tensor flops per algorithmic flop, so 1/3 = 0.333 of the "
                        "bf16 peak is this formulation's ceiling"
                        if impl == "tc" else "float32 SIMT FMA path (B200 fp32 vector peak ~74 TFLOP/s)",
                "stage_ms_per_step": dict({k: v / args.steps for k, v in stages.items()}, **other)}
        out = {"metric": "EI candidates/sec", "value": value, "unit": "candidates/s", "n_gpus": world,
               "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
               "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
               "data": "synthetic",
               "config": {"workload": "%s D=%d N=%d M=%d S=%d %s" % (args.workload, D, N, M, S, KIND),
                          "parallelism": "hyper-samples round-robin over %d GPU(s), one all-reduce of M floats" % world,
                          "l2": "working set (factors %.1f GB per rank) >> 126 MB L2, no flush needed"
                                % (Sl * (((N + 127) // 128) * 128) ** 2 * 4 / 1e9),
                          "pairs_per_sec": value * S, "argmax": int(idx.cpu()[0]), "argmax_e2e": best_idx},
               "e2e": {"value": M / (e2e_ms * 1e-3), "unit": "candidates/s", "ms_per_step": e2e_ms, "steps": args.steps,
                       "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                       "api": ("backend.grid_state + backend.ei_matrix (the calls GPEIperSecChooserB200 makes)" if per_s else
                               "GPEIOptChooserB200.ei_over_hypers(comp, pend, cand, vals)") +
                              " -> (M,S) float64 EI matrix on the host, host argmax of the mean"},
               "gpu_launches": launches, "clocks": clocks, "roofline": roof,
               "accuracy_guard": dict(eng.last_guard or {}, threshold=eng.guard_threshold)}
        if world == 1 and not args.no_cpu:
            cpu = cpu_port_sample(args.workload, D, N, M, S, budget_cands=args.cpu_cands)
            out["cpu_baseline"] = {"value": cpu["value"], "unit": "candidates/s", "cores": cpu["threads"],
                                   "kind": "port", "sample": cpu["sample"]}
            ref, got = cpu["ei"], ei_host[:cpu["Mc"], 0]        # sample 0 lives on rank 0 (column 0 of the matrix)
            out["parity"] = {"vs": "cpu_baseline sample (hyper-sample 0, first %d candidates)" % cpu["Mc"],
                             "parity_max_rel": float(np.abs(got - ref).max() / ref.max()),
                             "argmax_match": bool(int(np.argmax(got)) == int(np.argmax(ref))),
                             "tolerance": 5e-3}
            cpu.pop("ei")
        if world == 1 and not args.no_next and not per_s:
            out["next"] = next_wall_ms(args, D, N, M, S, backend)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_BYTES = 64 * 10 ** 6 - 4096          # 64 MB, less room for the .npy headers


def dump_outputs(path, arrays):
    """Writes each array as path/<name>.npy in float64.  When the EI matrix would take the total past DUMP_BYTES, a fixed
    seeded sample of its rows is written instead, with the row indices as ei_matrix_e2e_rows."""
    os.makedirs(path, exist_ok=True)
    mat = arrays["ei_matrix_e2e"]
    room = DUMP_BYTES - sum(a.nbytes for k, a in arrays.items() if k != "ei_matrix_e2e")
    if mat.nbytes > room:
        keep = room // (8 * (mat.shape[1] + 1)) - 1                  # float64 rows plus their float64 indices
        rows = np.sort(np.random.RandomState(0).choice(mat.shape[0], keep, replace=False))
        arrays = dict(arrays, ei_matrix_e2e=mat[rows], ei_matrix_e2e_rows=rows.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def next_wall_ms(args, D, N, M, S, backend):
    """Second half of BASELINE.json's metric: chooser.next() wall-ms through the plugin API at the benched workload
    (MCMC chain with the GPU float64 log-likelihood -> grid pass -> L-BFGS refinement with cached factors -> grid pass),
    steady state: burnin=0 stands for "second call" (the first call of a real run adds `burnin`=100 more sample_hypers).

    The CPU port of the same call is reported as counts x unit times (SURVEY 8d: the full reference next() at the
    headline size is multi-hour): log-likelihood evaluations x one O.gp_logprob, refinement evaluations x S x one
    O.grad_optimize_ei, two grid passes from the cpu_baseline fit.  --next-cpu runs the CPU port for real (small
    workloads only)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import next_bench
    calls = next_bench.run("gpu", D, N, M, S, burnin=0, calls=args.next_calls, grid_subset=20, backend=backend)
    last = calls[-1]
    out = {"workload": "%s D=%d N=%d M=%d S=%d burnin=0 (steady state) grid_subset=20" % (args.workload, D, N, M, S),
           "ms": float(np.mean([c["ms"] for c in calls])), "unit": "ms", "calls": len(calls),
           "phase_ms": last["phase_ms"], "loglik_evals": last["loglik_evals"], "loglik_batches": last["loglik_batches"],
           "refine_evals": last["refine_evals"]}
    if not args.no_cpu:
        from oracle import gp_oracle as O
        blas_threads()
        comp, cand, vals, hs = synth(D, N, M, S)
        pend = np.zeros((0, D))
        h = hs[0]
        O.gp_logprob(KIND, h[0], h[1], h[2], h[3], comp, vals)
        t0 = time.perf_counter()
        O.gp_logprob(KIND, h[0], h[1], h[2], h[3], comp, vals)
        t_ll = time.perf_counter() - t0
        t0 = time.perf_counter()
        O.grad_optimize_ei(KIND, h, cand[:1], comp, pend, vals)
        t_g = time.perf_counter() - t0
        grid = cpu_port_sample(args.workload, D, N, M, S, budget_cands=min(M, 2000))
        est = last["loglik_evals"] * t_ll + last["refine_evals"] * S * t_g + 2.0 * grid["t_full_s"]
        out["cpu_port_estimate"] = {
            "ms": 1e3 * est, "kind": "counts x unit times (extrapolation, not a timed run)",
            "loglik_unit_s": t_ll, "refine_eval_unit_s_per_sample": t_g, "grid_pass_s": grid["t_full_s"],
            "formula": "loglik_evals*t_loglik + refine_evals*S*t_grad + 2*t_grid_pass", "cores": _CORES}
        out["speedup_vs_cpu_port_estimate"] = (1e3 * est) / out["ms"]
    if args.next_cpu:
        cpu = next_bench.run("cpu", D, N, M, S, burnin=0, calls=1, grid_subset=20)
        out["cpu_port_ms_timed"] = cpu[-1]["ms"]
        out["cpu_cores"] = _CORES
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="headline", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-cands", type=int, default=None, help="candidates in the CPU sample")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--samples", type=int, default=None, help="override S (experiments only)")
    ap.add_argument("--no-next", action="store_true", help="skip the chooser.next() wall-ms leg")
    ap.add_argument("--next-calls", type=int, default=1, help="timed next() calls")
    ap.add_argument("--next-cpu", action="store_true", help="also run the CPU port of next() for real (slow)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's results of both EI legs to DIR/<name>.npy (float64, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    D, N, M, S = WORKLOADS[args.workload]
    if args.samples:
        S = args.samples
    if args.impl == "reference":
        run_reference_arm(args, D, N, M, S)
    else:
        run_b200_arm(args, D, N, M, S)


if __name__ == "__main__":
    main()
