#!/usr/bin/env python
"""bench.py — exact-GP log-marginal + gradient evaluations per second (fp64), the metric of BASELINE.json.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--n 16384] [--d 8] [--dump-outputs DIR]

One "step" = one evaluation (= one GP.parameters_changed(), GPy/core/gp.py:269-282): theta -> log marginal likelihood and
its gradient w.r.t. (variance, D lengthscales, noise) for GPRegression RBF ARD on the synthetic workload of
SURVEY.md §8(d) (BASELINE.json configs[1]: N=16384, D=8, fp64, 1xB200).

`value`  : evaluations/s with X, Y resident in HBM (theta in, (LML, grad) out each step), device-timed.
`e2e`    : the same metric through the reference-facing plugin API (gpy_b200.GPRegression over the C ABI) with HOST
           buffers: every step copies X and Y host->device and reads (LML, grad) back, inside the timed region.
`roofline`: dominant kernel = the digit-split int8 GEMM on the tcgen05 tensor cores (trailing update + K^-1); achieved = the
           int8 tensor operations it issues / its CUDA-event time, measured live over the timed steps; peak = 2 x the
           measured dense bf16 rate (MEASURED_PEAKS.json). On the fp64 DMMA path (option ozaki = 0, multi-GPU) the kernel
           is the DMMA GEMM and the peak the DMMA issue rate measured in the same run.
`cpu_baseline` / `--impl reference`: the reference's own CPU operation sequence (oracle/gpy_oracle.py: same LAPACK/BLAS
           calls incl. the wasted dtrtri, two exp passes, the serial ARD loop compiled from C) on this box's cores.
`--dump-outputs DIR`: after the timed steps, what the last timed step of each timed path returned to its caller is written
           as DIR/<name>.npy (float64; the largest, the sparse workload's gradient, has M x D + D + 2 entries). The inputs
           depend only on the arguments (fixed seeds), so two builds run with the same arguments can be compared output
           for output.
"""
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

METRIC = "exact-GP log-marginal+grad evals/sec (fp64) at N=16k D=8"
UNIT = "evals/s"


def synthetic(N, D, seed=0):
    """SURVEY.md §8(d) workload (same generator as oracle.gpy_oracle.synthetic, restated so the product arm does not
    import the oracle)."""
    rng = np.random.default_rng(seed)
    X = rng.uniform(-3, 3, (N, D))
    f = np.sin(X).sum(1, keepdims=True) / np.sqrt(D)
    Y = f + 0.1 * rng.standard_normal((N, 1))
    return X, Y


def theta_for_step(D, step):
    """theta_bench (variance 1, lengthscale sqrt(D), noise 0.01) perturbed deterministically per step, the way an
    optimizer iterate moves: nothing can be cached between steps."""
    rng = np.random.default_rng(1000 + step)
    var = 1.0 * (1.0 + 0.05 * rng.uniform(-1, 1))
    ls = np.sqrt(D) * (1.0 + 0.05 * rng.uniform(-1, 1, D))
    noise = 0.01 * (1.0 + 0.05 * rng.uniform(-1, 1))
    return var, ls, noise


class ClockSampler(object):
    """nvidia-smi sampler for the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, gpu_index=0):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(np.max(mx)), "power_w_max": float(np.max(power)),
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    """dense bf16 TFLOP/s (sustained) measured by the driver on this pool (MEASURED_PEAKS.json), else the fallback of
    B200_PROFILING.md (1.4 PFLOP/s sustained) -> (value, source)"""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            mp = json.load(f)
        return float(mp.get("bf16_tflops_sustained") or mp["bf16_tflops"]), "MEASURED_PEAKS.json (measured)"
    except Exception:
        return 1400.0, "B200_PROFILING.md fallback (1.4 PFLOP/s sustained bf16)"


def dump_outputs(args, arrays):
    """--dump-outputs DIR: each array as DIR/<name>.npy in float64"""
    if not args.dump_outputs:
        return
    os.makedirs(args.dump_outputs, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(args.dump_outputs, name + ".npy"), np.asarray(a, dtype=np.float64))


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ------------------------------------------------------------------------------------------------------------------
# reference arm: GPy's CPU operation sequence on the host cores
# ------------------------------------------------------------------------------------------------------------------
def cpu_eval_timed(N, D, step, native="port"):
    from oracle import gpy_oracle as o
    X, Y = synthetic(N, D)
    var, ls, noise = theta_for_step(D, step)
    t0 = time.perf_counter()
    lml, grad, _ = o.eval_lml_grad(X, Y, "rbf", True, var, ls, noise, native=native)
    return time.perf_counter() - t0, lml, grad


def cpu_threads():
    try:
        from threadpoolctl import threadpool_info
        infos = threadpool_info()
        return max([i.get("num_threads", 1) for i in infos] or [1]), infos
    except Exception:
        return os.cpu_count() or 1, []


def ensure_oracle_native():
    """build the checker's C helper if it is missing (the reference's serial Cython ARD loop, restated in C)."""
    so = os.path.join(ROOT, "oracle", "_build", "liboracle_c.so")
    if not os.path.exists(so):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "_build/liboracle_c.so"],
                              stdout=subprocess.DEVNULL)
    return "port"


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    native = ensure_oracle_native()
    N, D = args.n, args.d
    threads, infos = cpu_threads()
    for w in range(args.warmup):
        cpu_eval_timed(min(N, 2048), D, -1 - w, native)   # warm-up on a small instance: BLAS threads, page cache
    # Every step is one COMPLETE evaluation at the full size (no extrapolation); at N = 16384 one takes of the order of a
    # minute on the host cores.
    times = []
    t_start = time.perf_counter()
    for s in range(args.steps):
        dt, lml, grad = cpu_eval_timed(N, D, s, native)
        times.append(dt)
    total = time.perf_counter() - t_start
    per = float(np.mean(times))
    blas = ", ".join(sorted({"%s %s" % (i.get("internal_api"), i.get("version")) for i in infos}))
    line = {
        "impl": "reference", "metric": METRIC, "value": 1.0 / per, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(times), "warmup": args.warmup, "ms_per_step": per * 1e3,
        "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "GPRegression RBF ARD N=%d D=%d fp64 (BASELINE.json configs[1])" % (N, D),
                   "path": "GPy CPU operation sequence restated in oracle/gpy_oracle.py (GPy itself needs paramz, "
                           "absent from this image) and verified bit-identical to the unmodified GPy 1.14.2 "
                           "modules in the build container: dsyrk+symmetrify, 2 exp passes, dpotrf, dtrtri (unused), "
                           "dpotri, dpotrs, Cython helpers (symmetrify, serial ARD loop) restated in C, paramz caching "
                           "of r and K modelled"},
        "cpu_baseline": {"value": 1.0 / per, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "%d steps, each one complete evaluation at N=%d (warm-up at N=2048)" % (len(times), N),
                         "host_cpus": os.cpu_count(), "blas": blas},
        "e2e": {"value": 1.0 / per, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": total,
    }
    print(json.dumps(line), flush=True)
    dump_outputs(args, {"lml": lml, "grad": grad})


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    # rank 0 prints ONE JSON line on stdout: NCCL's own lines (version banner, INFO/INIT when NCCL_DEBUG asks for them)
    # are routed to stderr, not silenced — NCCL_DEBUG itself is left exactly as the caller set it
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    import torch
    import torch.distributed as dist
    rank, world, local = dist_env()
    N, D = args.n, args.d
    use_dist = world > 1
    torch.cuda.set_device(local)
    if use_dist:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from gpy_b200 import _ffi
    import gpy_b200

    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    X, Y = synthetic(N, D)
    eng = _ffi.Engine(local)
    # N > 1 GPUs. A matrix that fits one GPU is evaluated fastest by ONE GPU (the tcgen05 path is single-GPU; at N = 16384 one
    # B200 finishes an evaluation sooner than 2-8 GPUs sharing it, whose strong scaling is bound by the serial diagonal-block
    # chain and the per-panel collectives) — so for N <= 32768 the N GPUs run INDEPENDENT evaluations (different theta per
    # rank: multi-restart optimisation, the reference's own data-parallel pattern, paramz Model.optimize_restarts(parallel=
    # True)), no data-path collective, weak scaling; the sharded evaluation of the same size is measured and reported beside
    # it ("sharded_one_evaluation"). Beyond that size ONE evaluation is sharded over the GPUs (block-cyclic rows, NCCL).
    mode = args.mode if args.mode != "auto" else ("replicas" if N <= 32768 else "sharded")
    sharded = use_dist and mode == "sharded"
    if sharded:
        # ONE evaluation spread over all GPUs: block rows dealt block-cyclically, NCCL panel all-gathers (gpx_dist.cu)
        from gpy_b200 import dist as gdist
        gdist.init_engine_comm(eng)
    eng.set_data(X, Y)

    # ---- device-resident throughput ------------------------------------------------------------------------------
    for w in range(args.warmup):
        eng.exact_eval("rbf", True, *theta_for_step(D, -1 - w))
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = eng.total_launches()
    dev_ms, upd_ms, upd_flops, lau_ms, lau_flops, kb_ms, kb_bytes, upd_i8 = [], 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0
    upd_launches = 0
    barrier()
    t0 = time.perf_counter()
    last = None
    for s in range(args.steps):
        last = eng.exact_eval("rbf", True, *theta_for_step(D, s + (0 if sharded else 100000 * rank)))
        st = eng.stats()
        dev_ms.append(st["total_ms"])
        upd_ms += st["update_ms"]; upd_flops += st["update_flops"]; upd_launches += st["update_launches"]
        lau_ms += st["lauum_ms"]; lau_flops += st["lauum_flops"]
        kb_ms += st["kbuild_ms"]; kb_bytes += st["kbuild_bytes"]
        upd_i8 += st.get("update_int8_ops", 0.0)
    barrier()
    wall = time.perf_counter() - t0
    launches = eng.total_launches() - launches0
    clocks = sampler.stop() if rank == 0 else None
    t_dev = float(np.sum(dev_ms)) * 1e-3          # CUDA-event time of the K evaluations on the launching stream
    t_dev_t = torch.tensor([t_dev, wall], dtype=torch.float64, device="cuda")
    if use_dist:
        dist.all_reduce(t_dev_t, op=dist.ReduceOp.MAX)
    t_dev, wall = float(t_dev_t[0]), float(t_dev_t[1])
    # sharded: all ranks work on the same evaluation (strong scaling); replicas: one independent stream per GPU
    value = (1 if sharded or world == 1 else world) * args.steps / t_dev

    # ---- end to end through the plugin API with host buffers --------------------------------------------------------
    m = gpy_b200.GPRegression(X, Y, gpy_b200.RBF(D, ARD=True), noise_var=0.01, device=local, engine=eng)
    e2e_steps = args.steps
    m.update_model(False)                      # batch the writes: ONE parameters_changed() per step (set_theta)
    for w in range(min(args.warmup, 2)):
        m.set_XY(X.copy(), Y.copy())
        m.set_theta(*theta_for_step(D, -1 - w))
    barrier()
    t0 = time.perf_counter()
    e2e_dev_ms, e2e_setxy_ms = [], []
    for s in range(e2e_steps):
        ts = time.perf_counter()
        m.set_XY(X.copy(), Y.copy())           # fresh host buffers: forces the host->device copy of the inputs
        e2e_setxy_ms.append((time.perf_counter() - ts) * 1e3)
        m.set_theta(*theta_for_step(D, s))     # -> parameters_changed(): inference + kernel gradients
        ll = m.log_likelihood()
        g = m.gradient
        e2e_dev_ms.append(eng.stats()["total_ms"])
    barrier()
    e2e_wall = time.perf_counter() - t0
    if rank == 0:
        # device-resident path: (log marginal, gradient [variance, lengthscales.., noise], extra jitter) of the last step;
        # plugin API: log_likelihood() and gradient of its last step
        dump_outputs(args, {"lml": last[0], "grad": last[1], "jitter": last[2], "e2e_lml": ll, "e2e_grad": g})
    e2e_t = torch.tensor([e2e_wall], dtype=torch.float64, device="cuda")
    if use_dist:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_value = (1 if sharded or world == 1 else world) * e2e_steps / float(e2e_t[0])

    # ---- parity carried by the bench line itself when N > 1 (the driver's SCALE run has no other parity evidence) ---------
    parity_multi = None
    eng_s = eng if sharded else None
    if use_dist and not sharded:
        # the sharded evaluation of the same problem, timed the same way, for the record
        from gpy_b200 import dist as gdist
        eng_s = _ffi.Engine(local)
        gdist.init_engine_comm(eng_s)
        eng_s.set_data(X, Y)
        for w in range(2):
            eng_s.exact_eval("rbf", True, *theta_for_step(D, -1 - w))
        barrier()
        ms_s = []
        for s_ in range(args.steps):
            eng_s.exact_eval("rbf", True, *theta_for_step(D, s_))
            ms_s.append(eng_s.stats()["total_ms"])
        barrier()
        ts = torch.tensor([float(np.sum(ms_s)) * 1e-3], dtype=torch.float64, device="cuda")
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        sharded_side = {"value": args.steps / float(ts[0]), "unit": UNIT, "ms_per_step": float(ts[0]) / args.steps * 1e3,
                        "scaling": "strong", "parallelism": "%d GPUs, ONE evaluation sharded by block rows (memory-distributed, "
                        "block-cyclic), NCCL broadcast of the inverted diagonal block + all-gather of the panel, fp64 DMMA GEMMs" % world}
    if eng_s is not None and use_dist:
        th_last = theta_for_step(D, args.steps - 1)
        lml_s, grad_s, _ = eng_s.exact_eval("rbf", True, *th_last)    # collective: every rank takes part
        if rank == 0:
            e1 = _ffi.Engine(local)                                  # the single-GPU engine on the same device, same theta
            e1.set_data(X, Y)
            lml_1, grad_1, _ = e1.exact_eval("rbf", True, *th_last)
            e1.close()
            parity_multi = {"parity_vs_1gpu": {"lml_abs": abs(lml_s - lml_1),
                                               "grad_rel_max": float(np.max(np.abs(grad_s - grad_1) / np.abs(grad_1)))}}
            if N <= 4096:
                _, lml_c, grad_c = cpu_eval_timed(N, D, args.steps - 1, ensure_oracle_native())
                parity_multi["parity_vs_oracle"] = {"lml_abs": abs(lml_s - lml_c),
                                                    "grad_rel_max": float(np.max(np.abs(grad_s - grad_c) / np.abs(grad_c)))}
            if not sharded:
                sharded_side.update(parity_multi)
                parity_multi = {"sharded_one_evaluation": sharded_side}
        barrier()

    if rank == 0:
        peak = eng.measure_fp64_peak()
        cpu = None
        if world == 1 and not args.no_cpu:
            native = ensure_oracle_native()
            threads, infos = cpu_threads()
            cpu_eval_timed(2048, D, -1, native)
            dt, lml_c, grad_c = cpu_eval_timed(N, D, args.steps - 1, native)
            lml_g, grad_g, _ = last
            cpu = {"value": 1.0 / dt, "unit": UNIT, "cores": threads, "kind": "port",
                   "sample": "1 full evaluation at N=%d on the host cores (same theta as the last GPU step)" % N,
                   "seconds": dt, "host_cpus": os.cpu_count(),
                   "parity_vs_gpu": {"lml_abs": abs(lml_c - lml_g),
                                     "grad_rel_max": float(np.max(np.abs(grad_c - grad_g) / np.abs(grad_c)))}}
        nl = D
        whole = {"whole_eval_tflops_fp64": float(N) ** 3 * args.steps / t_dev * 1e-12,
                 "whole_eval_frac_of_dmma_peak": float(N) ** 3 * args.steps / t_dev * 1e-12 / (peak * (world if sharded else 1)) if peak else None,
                 "dmma_peak_tflops": peak,
                 "kbuild_gbs": kb_bytes / kb_ms * 1e-6 if kb_ms else None,
                 "share_of_step": upd_ms / (t_dev * 1e3) if t_dev else None,
                 "launches": (upd_launches / args.steps) if upd_launches else None}
        if upd_i8 > 0 and upd_ms > 0:
            # tcgen05 path: the dominant kernel is the int8 digit-split GEMM (trailing update + K^-1 in the same launches).
            # achieved = int8 tensor operations actually issued (2 per MAC, summed over the digit pairs computed: 36 per
            # fp64 product with 8 digits, 28 with 7) / CUDA-event time of those launches; peak = 2 x the measured dense bf16
            # rate of MEASURED_PEAKS.json (kind::i8 issues at exactly twice the kind::f16 rate on this part:
            # profiles/r02_microbench_tcgen05_i8_width_sweep.txt), the sustained figure because the kernel is timed inside a
            # long step.
            mp, src = measured_peaks()
            i8_peak = 2.0 * mp
            ach = upd_i8 / upd_ms * 1e-9
            roofline = {"bound": "tensor", "kernel": "oz_gemm2_kernel (tcgen05.mma kind::i8 digit-split GEMM, 128x128x32 MMAs in two "
                                                      "passes: trailing update + K^-1)",
                        "achieved": ach, "peak": i8_peak, "unit": "TFLOP/s", "frac": ach / i8_peak,
                        "unit_note": "int8 tensor operations (2 per multiply-add), not floating point",
                        "peak_source": "2 x bf16_tflops_sustained of %s" % src,
                        # for context: the kind::i8 ISSUE rate of this part (8192 MAC/clk/SM, tools/microbench_tcgen05.cu) at the
                        # SM clock sampled during this run; cuBLAS bf16 itself reaches ~0.73 of the corresponding bf16 issue rate
                        "frac_of_i8_issue_rate": ach / (2 * 8192 * 148 * (clocks["sm_mhz"] or 1965.0) * 1e-6)
                        if clocks and clocks.get("sm_mhz") else None,
                        "fp64_equivalent_tflops": upd_flops / upd_ms * 1e-9,
                        "algorithmic_flops_per_step": upd_flops / args.steps,
                        "traffic": None,
                        "traffic_note": "not measured in this run; per-launch DRAM traffic differs launch to launch (16 panels): the ncu "
                                        "capture of the same path (profiles/r02s3_final_oz_traffic.txt) has 2.61 GB per large launch "
                                        "(1.8 GB read + 0.9 GB written) at N=16384",
                        "grad_from_kinv_ms_per_step": lau_ms / args.steps}
        else:
            ach = upd_flops / upd_ms * 1e-9 if upd_ms > 0 else 0.0
            roofline = {"bound": "tensor", "kernel": "gemm_update_kernel (fp64 DMMA trailing update)",
                        "achieved": ach if upd_ms > 0 else None, "peak": peak, "unit": "TFLOP/s",
                        "frac": ach / peak if (peak and upd_ms > 0) else None,
                        "note": None if upd_ms > 0 else "per-kernel event accounting is single-GPU; see whole_eval_*",
                        "traffic": None,
                        "peak_source": "fp64 DMMA.8x8x4 issue rate measured in this run (gpx_measure_fp64_peak); "
                                       "MEASURED_PEAKS.json holds no fp64 entry",
                        "lauum_tflops": lau_flops / lau_ms * 1e-9 if lau_ms else None}
        roofline.update(whole)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t_dev / args.steps * 1e3, "higher_is_better": True,
            # per-GPU work is fixed as N grows (one evaluation stream per GPU) unless ONE evaluation is sharded; the N = 1
            # line carries the same label as the N > 1 lines it is compared with
            "scaling": "strong" if (sharded or mode == "sharded") else "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": "GPRegression RBF ARD N=%d D=%d fp64 (BASELINE.json configs[1])" % (N, D),
                       "theta": "theta_bench (variance 1, lengthscale sqrt(D), noise 0.01) +-5% per step",
                       "parallelism": "1 GPU" if world == 1 else (
                           "%d GPUs, one evaluation sharded by block rows (memory-distributed, block-cyclic), NCCL broadcast + "
                           "all-gather of panels" % world if sharded else
                           "%d GPUs, one independent evaluation stream per GPU (different theta per rank, no data-path "
                           "collective); the sharded evaluation of the same size is in sharded_one_evaluation" % world),
                       "l2": "inputs larger than L2: the %.1f GiB workspace is rebuilt and streamed every step"
                             % (N * N * 8 / 2**30),
                       "timing": "CUDA events on the launching stream around each evaluation, max over ranks"},
            "wall_ms_per_step": wall / args.steps * 1e3,
            "gpu_launches": int(launches),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(X.nbytes + Y.nbytes + (D + 2) * 8),
                    "d2h_bytes_per_step": int((nl + 3) * 8), "steps": e2e_steps,
                    "device_ms_per_step": float(np.mean(e2e_dev_ms)), "set_XY_host_ms_per_step": float(np.mean(e2e_setxy_ms)),
                    "api": "gpy_b200.GPRegression.set_XY/set_theta -> log_likelihood(), gradient (host ndarrays in/out)"},
            "roofline": roofline,
            "cpu_baseline": cpu,
            "clocks": clocks,
        }
        if parity_multi:
            line.update(parity_multi)
        print(json.dumps(line), flush=True)
    if use_dist:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------------
# --workload sparse: BASELINE.json configs[4] (SparseGPRegression RBF N=262144 M=4096 D=16), one VarDTC evaluation per step
# ------------------------------------------------------------------------------------------------------------------
def run_sparse(args):
    """One step = one SparseGP.parameters_changed() (GPy/core/sparse_gp.py:76-119: VarDTC bound + all gradients incl. dZ)
    through gpy_b200.SparseGPRegression over the C ABI. value = device-resident evaluations/s (X, Y in HBM; Z and theta
    in, bound and gradients out), e2e = the same with X, Y re-uploaded from the host every step."""
    import torch
    rank, world, local = dist_env()
    if world > 1 and rank != 0:
        return                                   # replicas only: the driver's line comes from rank 0 (row sharding: tools/)
    torch.cuda.set_device(local)
    import gpy_b200
    N, M, D = args.n if args.n != 16384 else 262144, args.m, args.d if args.d != 8 else 16
    rng = np.random.default_rng(0)
    X = rng.uniform(-3, 3, (N, D))
    Y = np.sin(X).sum(1, keepdims=True) / np.sqrt(D) + 0.1 * rng.standard_normal((N, 1))
    Z = X[rng.permutation(N)[:M]].copy()         # sparse_gp_regression.py:41-43: a random subset of the inputs
    ls0 = np.full(D, np.sqrt(D))
    k = gpy_b200.RBF(D, variance=1.0, lengthscale=ls0, ARD=True)
    m = gpy_b200.SparseGPRegression(X, Y, kernel=k, Z=Z, device=local)
    eng = m.inference_method.engine

    def step(i, reupload):
        r = np.random.default_rng(2000 + i)
        if reupload:
            m.inference_method.invalidate_data()
        k.variance.values[...] = 1.0 * (1 + 0.05 * r.uniform(-1, 1))
        k.lengthscale.values[...] = ls0 * (1 + 0.05 * r.uniform(-1, 1, D))
        m.likelihood.variance.values[...] = 0.05 * (1 + 0.05 * r.uniform(-1, 1))
        m.parameters_changed()
        return m.log_likelihood()

    for w in range(args.warmup):
        step(-1 - w, False)
    sampler = ClockSampler(local)
    sampler.start()
    l0 = eng.total_launches()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(i, False)
    torch.cuda.synchronize()
    t_res = time.perf_counter() - t0
    last = {"lml": m.log_likelihood(), "grad": m.gradient}     # gradient: [Z (M x D, row-major), variance, lengthscales.., noise]
    launches = eng.total_launches() - l0
    clocks = sampler.stop()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(i, True)
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    dump_outputs(args, dict(last, e2e_lml=m.log_likelihood(), e2e_grad=m.gradient))
    flops = 4.0 * N * M * M + 20.0 * M ** 3       # DESIGN.md §7b: tmp, A, dL_dKnm over N M^2 + the M x M algebra
    peak = eng.measure_fp64_peak()
    ach = flops * args.steps / t_res * 1e-12
    cpu = None
    if not args.no_cpu:
        from oracle import gpy_oracle as o
        Ns = min(N, 16384)                         # bounded sample: the first Ns rows, same Z / theta (CPU work is ~ linear in N)
        ts = time.perf_counter()
        lml_c, g_c, Zg_c, _ = o.sparse_eval(X[:Ns], Y[:Ns], Z, "rbf", True, 1.0, ls0, 0.05)
        dt = time.perf_counter() - ts
        threads, _ = cpu_threads()
        cpu = {"value": 1.0 / (dt * N / Ns), "unit": "evals/s", "cores": threads, "kind": "port",
               "sample": "oracle VarDTC (var_dtc.py:66-276 restated) on the first %d of %d rows, same Z and theta: %.1f s, "
                         "scaled by N/Ns (the N-dependent work is linear in N)" % (Ns, N, dt), "seconds_sample": dt}
        try:   # parity of the device evaluation on the SAME sample (outside the timed regions; never breaks the line)
            e2 = gpy_b200._ffi.Engine(local)
            e2.sparse_set_data(X[:Ns], Y[:Ns])
            lml_g, g_g, Zg_g = e2.sparse_eval("rbf", True, 1.0, ls0, Z, 0.05)
            e2.close()
            cpu["parity_vs_gpu_on_sample"] = {
                "lml_rel": abs(lml_g - lml_c) / max(1.0, abs(lml_c)),
                "grad_rel_max": float(np.max(np.abs(g_g - g_c) / np.maximum(np.abs(g_c), 1e-300))),
                "dZ_max_over_largest": float(np.max(np.abs(Zg_g - Zg_c)) / max(float(np.abs(Zg_c).max()), 1e-300))}
        except Exception as ex:  # noqa: BLE001
            cpu["parity_vs_gpu_on_sample"] = {"error": repr(ex)}
    line = {"metric": "SparseGPRegression VarDTC bound+gradient evals/sec (fp64) at N=%d M=%d D=%d" % (N, M, D),
            "value": args.steps / t_res, "unit": "evals/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t_res / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "SparseGPRegression RBF ARD N=%d M=%d D=%d (BASELINE.json configs[4])" % (N, M, D),
                       "l2": "inputs larger than L2: psi1 = K(X, Z) is %.1f GB and is rebuilt every step" % (8.0 * N * M / 1e9),
                       "timing": "host clock around K steps with a device synchronize on both sides (one process)"},
            "gpu_launches": int(launches),
            "e2e": {"value": args.steps / t_e2e, "unit": "evals/s", "h2d_bytes_per_step": int(X.nbytes + Y.nbytes + Z.nbytes),
                    "d2h_bytes_per_step": int((D + 3 + M * D) * 8),
                    "api": "gpy_b200.SparseGPRegression.parameters_changed() with the data re-uploaded every step"},
            "roofline": {"bound": "tensor", "kernel": "gemm_panel_kernel (fp64 DMMA, the three N M^2 products)", "achieved": ach,
                         "peak": peak, "unit": "TFLOP/s", "frac": ach / peak if peak else None, "traffic": None,
                         "algorithmic_flops_per_step": flops,
                         "peak_source": "fp64 DMMA issue rate measured in this run"},
            "cpu_baseline": cpu, "clocks": clocks, "lml_last": float(m.log_likelihood())}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps (>= 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", "--n", dest="n", type=int, default=16384, help="number of data points N")
    ap.add_argument("--d", type=int, default=8)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--workload", default="exact", choices=["exact", "sparse"],
                    help="exact = BASELINE.json configs[1] (the metric); sparse = configs[4] (VarDTC, N=262144 M=4096 D=16)")
    ap.add_argument("--m", type=int, default=4096, help="inducing points (sparse workload)")
    ap.add_argument("--mode", default="auto", choices=["auto", "sharded", "replicas"],
                    help="N>1 GPUs: auto = independent evaluations per GPU while the matrix fits one GPU (N <= 32768), one "
                         "sharded evaluation beyond; or force either")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "sparse":
        run_sparse(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
