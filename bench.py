#!/usr/bin/env python
"""bench.py - hypothesis x point evaluations per second and ms per robust fit of the USAC hypothesize-and-verify path.

Workload (BASELINE.json configs[1]): homography, 4-point normalized DLT, inlier count + error sum (MSAC derivable),
uniform sampler, N = 4000 correspondences, 30 % inliers, threshold 2 px, confidence 0.95, max 10 000 iterations.
One such fit is ~1.5 M evaluations (a few microseconds of B200 time), so a "step" is a BATCH of independent image
pairs of that size - the reference's own batched use (Tests::getStatisticalResults loops fits, test/tests.h:148-150) -
all run to their own adaptive termination through usac_gpu_fit (sample -> solve -> score -> best-update -> terminate).

  value : useful evaluations/s with the point sets resident in HBM. "Useful" = the evaluations the sequential loop of
          ransac.cpp:58-139 executes for the same sample stream (speculative tail of the last round is NOT counted).
          One context, one stream. (`config.value_pipelined`: the step split over --pipe contexts/streams, for information.)
  e2e   : the same with HOST buffers: every step copies the step's point sets host->device (pinned memory) through
          usac_gpu_set_points, fits, and reads the results (model, inliers, score, iterations) back; the step is split
          over --pipe parts, each double-buffered (two contexts), so that uploads overlap the fits of other parts/steps.
  roofline : the scoring kernel, FP32 bound (BASELINE.json: "the roofline is FP32 FMA throughput plus HBM point
          streaming"); algorithmic 42 flop per homography evaluation (SURVEY.md section 8d).
  cpu_baseline / --impl reference : the reference's own Ransac::run compiled from its sources (oracle/_ref, built in the
          development container by oracle/Makefile.ref and shipped prebuilt; kind "reference") on the box's host cores, on a
          bounded sample of the same problems; the oracle restatement (kind "port") when that library is absent.

Multi-GPU: one process per GPU (torchrun); independent image pairs shard across ranks with no data-path collective
(weak scaling: every rank owns --problems pairs). `--workload c5` instead shards the HYPOTHESES of one 1M-point fit
across the ranks with one NCCL all-gather per round (BASELINE.json configs[4]).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FLOPS_PER_EVAL = {"homography": 42, "fundamental": 33, "essential": 44, "line2d": 4}   # SURVEY.md section 8d
THR, CONF, MAX_IT, N_POINTS, INLIER_RATIO = 2.0, 0.95, 10000, 4000, 0.3
METRIC = "hypothesis x point evaluations/s (useful, whole job); ms per robust fit in config"


def env_int(name, default):
    return int(os.environ.get(name, default))


def make_problems(count, first_seed):
    from ransac_b200 import generator as gen
    return [gen.homography(n=N_POINTS, inlier_ratio=INLIER_RATIO, seed=first_seed + i)[0] for i in range(count)]


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, fields):
    """--dump-outputs: what the timed path returned for its last step, one DIR/<field>.npy per result field with one row per
    fit, so that two builds can be compared output for output. float32 fields stay float32, integer fields are written as
    float64 (exact below 2**53). Rows beyond 64 MB in all are sampled (fixed seed, ascending) and rows.npy names the kept ones."""
    arrays = {k: np.asarray(v, np.float32 if np.asarray(v).dtype == np.float32 else np.float64) for k, v in fields.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a[:1].nbytes for a in arrays.values()) + 8
    budget = DUMP_LIMIT - 256 * (len(arrays) + 1)          # room for the .npy headers
    if n * row_bytes > budget:
        keep = np.sort(np.random.default_rng(0).choice(n, budget // row_bytes, replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
        arrays["rows"] = keep.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def record_fields(rec):
    """usac_fit_result records (GpuContext.fit_records) -> {field: array}."""
    return {k: rec[k] for k in rec.dtype.names}


# ---------------------------------------------------------------------------------------------------------------------
# clocks sampler (NVML): SM clock + throttle reasons during the timed region
# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.samples, self.reasons, self.stop_flag, self.thread, self.max_mhz = [], set(), False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:   # noqa: BLE001
            self.nv, self.err = None, str(e)

    def _run(self):
        while not self.stop_flag:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:   # noqa: BLE001
                pass
            time.sleep(0.02)

    def start(self):
        if self.nv:
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "no NVML samples"}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle on the host cores
# ---------------------------------------------------------------------------------------------------------------------
def ref_available():
    """oracle/_ref/libusac_ref.so: the reference's own usac/ sources compiled in the development container (oracle/Makefile.ref);
    it travels to the GPU box as a prebuilt file. Without it the CPU arm falls back to the oracle port."""
    try:
        from oracle import ref as R
        R.lib()
        return True
    except Exception:   # noqa: BLE001
        return False


def cpu_fits(problems, seeds, threads, impl="port"):
    """-> (evals, seconds, results) of CPU fits over `problems`, independent fits spread over `threads` host threads.
    impl "reference": Ransac::Ransac + Ransac::run of the compiled reference (evals = main-loop iterations x N, the scoring work
    of ransac.cpp:97; the refit loop's <= 8 x N evaluations are not counted); "port": the oracle restatement."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import oracle as O
    O.lib()
    if impl == "reference":
        from oracle import ref as R

        def one(args):
            p, s = args
            r = R.ransac_run(O.EST_HOMOGRAPHY, p, THR, conf=CONF, max_it=MAX_IT, seed=s)
            r["evals"] = int(r["iterations"]) * len(p)
            return r
    else:
        def one(args):
            p, s = args
            return O.ransac(p, O.EST_HOMOGRAPHY, rng=O.RNG_PHILOX, threshold=THR, confidence=CONF, max_iterations=MAX_IT, seed=s)
    t0 = time.perf_counter()
    if threads == 1:
        rs = [one(a) for a in zip(problems, seeds)]
    else:
        with ThreadPoolExecutor(threads) as ex:
            rs = list(ex.map(one, zip(problems, seeds)))
    dt = time.perf_counter() - t0
    return sum(r["evals"] for r in rs), dt, rs


REF_SAMPLE_NOTE = ("oracle/_ref/libusac_ref.so = the reference's own usac/ sources (Ransac::run, HomographyEstimator::GetError, DLT4p ...) compiled "
                   "-O2 -ffp-contract=off with stand-in OpenCV headers; its 4-point solver takes the wrong row of a thin SVD (dlt.cpp:43-48), so its "
                   "termination criterion never fires and every fit runs max_iter iterations - the metric is evaluations per second either way")


def cpu_baseline(budget_s=12.0):
    """Bounded sample: as many C2 problems as fit ~budget_s of wall time on all host cores (the reference itself is
    single-threaded; the per-core figure is reported next to it)."""
    cores = os.cpu_count() or 1
    impl = "reference" if ref_available() else "port"
    probe = make_problems(2, 5000)
    e1, t1, _ = cpu_fits(probe, [1, 1], 1, impl)
    per_fit = t1 / 2
    count = int(max(cores, min(4096, budget_s / per_fit * cores * 0.8)))
    problems = make_problems(count, 1000)
    evals, dt, rs = cpu_fits(problems, [1] * count, cores, impl)
    out = {"value": evals / dt, "unit": "evals/s", "cores": cores, "kind": impl,
           "sample": f"{count} of the C2 image pairs (first seeds of the GPU batch), {cores} threads over independent fits; single thread: "
                     f"{e1 / t1:.3e} evals/s. " + (REF_SAMPLE_NOTE if impl == "reference" else "oracle/libusac_oracle.so (restatement) -O2 -ffp-contract=off"),
           "ms_per_fit": dt / count * 1e3, "single_thread_value": e1 / t1}
    if impl == "reference":     # the oracle port beside it, for information (it terminates adaptively like the GPU path)
        ep, tp, _ = cpu_fits(problems[:max(cores, 64)], [1] * max(cores, 64), cores, "port")
        out["oracle_port_value"] = ep / tp
    return out


def run_reference_arm(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    impl = "reference" if ref_available() else "port"
    per_step = max(cores, args.ref_problems if impl == "port" else min(args.ref_problems, 2 * cores))
    problems = make_problems(per_step, 1000)
    seeds = [1] * per_step
    for _ in range(args.warmup if impl == "port" else min(args.warmup, 1)):
        cpu_fits(problems[:cores], seeds[:cores], cores, impl)
    evals = 0
    t = 0.0
    for _ in range(args.steps):
        e, dt, rs = cpu_fits(problems, seeds, cores, impl)
        evals += e
        t += dt
    v = evals / t
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: [r[k] for r in rs] for k in rs[0] if np.asarray(rs[0][k]).dtype.kind in "biuf"})
    sample = (f"{per_step} C2 image pairs per step, all host threads over independent fits; " +
              (REF_SAMPLE_NOTE if impl == "reference" else "CPU oracle (restated reference), oracle/libusac_oracle.so"))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "evals/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(per_step), "problems_per_step": per_step, "ms_per_fit": t / args.steps / per_step * 1e3},
            "cpu_baseline": {"value": v, "unit": "evals/s", "cores": cores, "kind": impl, "sample": sample},
            "e2e": {"value": v, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_name(problems=None):
    """Identical for the GPU arm and the reference arm (the driver compares the strings); the number of image pairs per step -
    the full batch on the GPU, a bounded sample of it on the CPU - is `config.problems_per_step`."""
    return (f"C2 homography 4-pt normalized DLT, uniform sampler, N={N_POINTS}, {int(INLIER_RATIO * 100)}% inliers, thr {THR}, "
            f"conf {CONF}, max_iter {MAX_IT}; step = a batch of independent image pairs per GPU, each run to adaptive termination")


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
def run_native(args):
    import torch
    import torch.distributed as dist

    from ransac_b200 import GpuContext, capi
    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    from ransac_b200 import dist as D0
    # several ranks on one host: bind each to the CPUs next to its GPU before any pinned allocation (staging buffers on the GPU's own
    # NUMA node); a single rank keeps every host core (the cpu_baseline leg uses them)
    numa_cpus = D0.bind_to_gpu_numa(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    B = args.problems
    problems = make_problems(B, 1000 + rank * B)
    host = torch.empty((B * N_POINTS, 4), dtype=torch.float32).pin_memory()
    host.numpy()[:] = np.concatenate(problems)
    sizes = [N_POINTS] * B

    ctx = GpuContext(local)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    info = ctx.device_info()
    fit_kw = dict(threshold=THR, confidence=CONF, max_iterations=MAX_IT, seed=1, round_size=args.round_size)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, steps):
        """K steps bracketed by barrier+synchronize, CUDA events on the launching stream -> (ms, per-step stats)."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stats = []
        barrier()
        with torch.cuda.stream(stream):
            ev0.record(stream)
            for _ in range(steps):
                stats.append(step_fn())
            ev1.record(stream)
        barrier()
        return ev0.elapsed_time(ev1), stats

    last = [None]          # the records of the latest resident step (--dump-outputs)

    def step_resident():
        res = last[0] = ctx.fit_records(**fit_kw)
        t = ctx.last_timing()
        return (int(res["useful_evals"].sum()), int(res["evals"].sum()), t["launches"], t["score_launches"], t["score_ms"],
                int(res["iterations"].sum()), int(res["rounds"].max()), int(res["rounds"].sum()))

    # e2e: the public API with HOST buffers. n_pipe contexts (streams, host threads) each own a share of the step's image pairs,
    # so that the host->device copy of one share overlaps the fits of the others (the copy engine and the SMs run
    # concurrently); every step still uploads every point set and reads every result back.
    n_pipe = max(1, min(args.pipe, B))
    halves = [(i * B // n_pipe, (i + 1) * B // n_pipe) for i in range(n_pipe)]
    pipe_ctx, pipe_streams = [], []
    for _ in range(n_pipe):
        c2 = GpuContext(local)
        s2 = torch.cuda.Stream()
        c2.set_stream(s2.cuda_stream)
        pipe_ctx.append(c2)
        pipe_streams.append(s2)

    # second buffer set for the e2e arm: part i owns contexts pipe_ctx[i] and pipe_ctx2[i]; one is being uploaded into while
    # the other one is being fitted (a lock per part keeps the two fits of a part from running at once)
    pipe_ctx2 = []
    for _ in range(n_pipe):
        c2 = GpuContext(local)
        s2 = torch.cuda.Stream()
        c2.set_stream(s2.cuda_stream)
        pipe_ctx2.append(c2)
        pipe_streams.append(s2)
    part_locks = [threading.Lock() for _ in range(n_pipe)]

    def e2e_part(cx, i, out, k):
        torch.cuda.set_device(local)
        lo, hi = halves[i]
        cx.set_points(capi.EST_HOMOGRAPHY, host[lo * N_POINTS:hi * N_POINTS], sizes[lo:hi])      # H2D of this step's points + re-layout
        with part_locks[i]:
            res = cx.fit_records(**fit_kw)
            t = cx.last_timing()
        out[k] = (int(res["useful_evals"].sum()), int(res["evals"].sum()), t["launches"], t["score_launches"], t["score_ms"],
                  int(res["iterations"].sum()), int(res["rounds"].max()))

    def timed_e2e(steps):
        """2 x n_pipe worker threads: part i of every step (1/n_pipe of the image pairs) is handled alternately by two threads
        with their own context/stream, each doing upload -> fit -> read back; while one of them fits step k the other uploads
        step k+1. The bracket is a pair of events on an idle timing stream recorded after a full device sync on each side, so
        all the work of the `steps` steps (every upload, every fit, every result read-back) lies between them."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        outs = [[None] * steps for _ in range(n_pipe)]

        def worker(i, j):
            cx = (pipe_ctx, pipe_ctx2)[j][i]
            for k in range(j, steps, 2):
                e2e_part(cx, i, outs[i], k)
        barrier()
        ev0.record(stream)
        threads = [threading.Thread(target=worker, args=(i, j)) for i in range(n_pipe) for j in range(2)]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
        torch.cuda.synchronize()
        ev1.record(stream)
        barrier()
        stats = [tuple(sum(outs[i][k][f] for i in range(n_pipe)) if f != 6 else max(outs[i][k][f] for i in range(n_pipe)) for f in range(7))
                 for k in range(steps)]
        return ev0.elapsed_time(ev1), stats

    def resident_part(i, out):
        torch.cuda.set_device(local)
        res = pipe_ctx[i].fit_records(**fit_kw)
        t = pipe_ctx[i].last_timing()
        out[i] = (int(res["useful_evals"].sum()), int(res["evals"].sum()), t["launches"], t["score_launches"], t["score_ms"],
                  int(res["iterations"].sum()), int(res["rounds"].max()))

    def step_resident_pipelined():
        out = [None] * n_pipe
        threads = [threading.Thread(target=resident_part, args=(i, out)) for i in range(n_pipe)]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
        return tuple(sum(o[k] for o in out) if k != 6 else max(o[k] for o in out) for k in range(7))

    def timed_threads(step_fn, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stats = []
        barrier()
        ev0.record(stream)
        for _ in range(steps):
            stats.append(step_fn())
        torch.cuda.synchronize()
        ev1.record(stream)
        barrier()
        return ev0.elapsed_time(ev1), stats

    # ---- device-resident arm ----
    # (a) one context, one stream: the reported `value`, and the per-launch CUDA-event times of the scoring kernel (roofline);
    # (b) for information, the same step split over --pipe contexts/streams (config.value_pipelined). The scoring kernel is
    #     persistent and fills every SM, so the small kernels of another stream cannot run beside it: splitting the step only
    #     makes the launches smaller. (Up to kernel v4 the static work split left long tails and (b) was the faster arm.)
    ctx.set_points(capi.EST_HOMOGRAPHY, host, sizes)
    timed(step_resident, args.warmup)
    clocks = ClockSampler(local)
    clocks.start()
    ms, stats = timed(step_resident, args.steps)
    clk = clocks.stop()
    ms_single = ms
    resident_out = last[0]
    for i, (lo_, hi_) in enumerate(halves):
        pipe_ctx[i].set_points(capi.EST_HOMOGRAPHY, host[lo_ * N_POINTS:hi_ * N_POINTS], sizes[lo_:hi_])
    timed_threads(step_resident_pipelined, args.warmup)
    ms_pipe, stats_p = timed_threads(step_resident_pipelined, args.steps)
    useful = sum(s[0] for s in stats)
    executed_p = sum(s[1] for s in stats)
    launches = sum(s[2] for s in stats)
    iters = sum(s[5] for s in stats)
    executed = executed_p
    score_launches = sum(s[3] for s in stats)
    score_ms = sum(s[4] for s in stats)
    # ---- end-to-end arm (host buffers) ----
    timed_e2e(2)
    ms_e2e, stats_e2e = timed_e2e(args.steps)
    useful_e2e = sum(s[0] for s in stats_e2e)
    # the upload alone, all ranks at once (what the host memory system and the PCIe tree give `world` GPUs together): the floor of an
    # end-to-end step, since every step uploads every point set
    scratch = torch.empty_like(host, device="cuda")
    evu0, evu1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        scratch.copy_(host, non_blocking=True)
        barrier()
        evu0.record(stream)
        for _ in range(5):
            scratch.copy_(host, non_blocking=True)
        evu1.record(stream)
    barrier()
    h2d_only_ms = evu0.elapsed_time(evu1) / 5
    del scratch
    # results: one 176-byte FitState record per problem at the end + one `done` int per still-active problem per round
    d2h_step = B * 176 + sum(s[6] for s in stats_e2e) / args.steps * B * 4   # (upper bound: every problem active in every round)

    # ---- second leg: the hypothesis-sharded 1M-point fit (config.c5) ----
    c5 = None
    if not args.no_c5:
        for c2 in pipe_ctx + pipe_ctx2:
            c2.close()
        pipe_ctx, pipe_ctx2 = [], []
        c5 = c5_leg(args, rank, world, local, args.steps, 3)

    h2d_all = torch.tensor([h2d_only_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(h2d_all, op=dist.ReduceOp.MAX)
    h2d_only_ms = float(h2d_all.item())
    t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([useful, useful_e2e, executed_p, launches], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    ms_all, ms_e2e_all = t.tolist()
    useful_all, useful_e2e_all, executed_all, launches_all = cnt.tolist()

    if rank == 0:
        fp32_nominal = 2.0 * 128 * info["sm_count"] * info["sm_clock_khz"] * 1e3 / 1e12    # TFLOP/s at the max SM clock
        measured_ffma = ctx.measure_fp32_peak()
        # MEASURED_PEAKS.json carries HBM and bf16 figures only: the FP32 denominator is MEASURED in this run (a register-resident
        # FFMA loop on every SM, usac_gpu_measure_fp32_peak), the nominal 2 x 128 lanes x SMs x max clock is kept beside it
        fp32_peak = measured_ffma if measured_ffma > 0 else fp32_nominal
        peak_source = (f"measured in this run: register-resident FFMA loop, {measured_ffma:.1f} TFLOP/s (nominal 2*128 lanes*SMs*max SM clock = "
                       f"{fp32_nominal:.1f}; MEASURED_PEAKS.json has no FP32 figure)")
        flops_launch = FLOPS_PER_EVAL["homography"] * executed / max(score_launches, 1)
        ach = flops_launch / (score_ms / max(score_launches, 1) * 1e-3) / 1e12
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:   # noqa: BLE001
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        # HBM side of one launch: the points of every image pair still active in that round once (16 B per point) + one
        # 128-byte record per model scored; sum(rounds) over the fits = number of (image pair, launch) incidences
        pair_launches = sum(s[7] for s in stats)
        alg_bytes_launch = (16.0 * N_POINTS * pair_launches + 128.0 * executed / N_POINTS) / max(score_launches, 1)
        traffic, traffic_note = None, None
        pipe = None
        try:   # DRAM bytes of one ncu --set full capture of this kernel (profiles/): a full-size launch, not this run's average
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
            pipe = tj.get("fma_pipe_pct")
            traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
            traffic_note = f"{tj['launch']}: {traffic / 1e6:.1f} MB DRAM vs {tj['algorithmic_bytes'] / 1e6:.1f} MB algorithmic ({tj['source']})"
        except Exception:   # noqa: BLE001
            pass
        roofline = {"bound": "fp32", "kernel": "score_sq_kernel<HOMOGRAPHY>", "achieved": ach, "peak": fp32_peak, "unit": "TFLOP/s",
                    "frac": ach / fp32_peak, "traffic": traffic, "traffic_note": traffic_note,
                    "fma_pipe_busy_pct_ncu": pipe,
                    "peak_source": peak_source, "peak_nominal": fp32_nominal, "frac_of_nominal": ach / fp32_nominal,
                    "flops_per_eval": 42, "evals_per_launch": executed / max(score_launches, 1),
                    "note": "achieved = ALGORITHMIC flops (42 per evaluation, the reference's formulation) / launch time. The kernel is exact but does "
                            "less arithmetic than that: a division-free forward test proves most evaluations outliers; the rest is re-evaluated with "
                            "the reference's arithmetic from a per-warp survivor queue. fma_pipe_busy_pct_ncu is the hardware-side figure (ncu capture, profiles/)",
                    "avg_launch_ms": score_ms / max(score_launches, 1), "score_share_of_step": score_ms / ms_single,
                    "hbm": {"algorithmic_bytes_per_launch": alg_bytes_launch,
                            "achieved_gbs": alg_bytes_launch / (score_ms / max(score_launches, 1) * 1e-3) / 1e9,
                            "peak_gbs": hbm_peak, "peak_source": "measured" if peaks else "fallback"}}
        line = {"metric": METRIC, "value": useful_all / (ms_all * 1e-3), "unit": "evals/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_all / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload_name(B), "problems_per_step": B, "problems_per_gpu": B, "round_size": args.round_size,
                           "l2": f"inputs larger than L2: {B * N_POINTS * 32 / 1e6:.0f} MB of points per GPU (AoS + pair layout) vs 126 MB",
                           "ms_per_fit": ms_all / args.steps / B, "avg_iterations_per_fit": iters / (args.steps * B),
                           "value_pipelined": sum(s[0] for s in stats_p) / (ms_pipe * 1e-3), "pipelined_streams": n_pipe,
                           "evals_executed_per_s": executed_all / (ms_all * 1e-3), "useful_fraction": useful / max(executed_p, 1)},
                "clocks": clk, "gpu_launches": int(launches_all),
                "e2e": {"value": useful_e2e_all / (ms_e2e_all * 1e-3), "unit": "evals/s", "h2d_bytes_per_step": B * N_POINTS * 16,
                        "d2h_bytes_per_step": int(d2h_step), "ms_per_step": ms_e2e_all / args.steps, "ms_per_fit": ms_e2e_all / args.steps / B,
                        "h2d_only_ms_per_step": h2d_only_ms, "h2d_only_gb_per_s_per_gpu": B * N_POINTS * 16 / (h2d_only_ms * 1e-3) / 1e9,
                        "h2d_note": "the step's uploads alone, all ranks at once (max over ranks): the floor of an end-to-end step; "
                                    "ranks are bound to the CPUs next to their GPU before pinned memory is allocated: " + str(numa_cpus)},
                "roofline": roofline}
        if c5 is not None:
            line["config"]["c5"] = c5
        if not args.no_epipolar:
            line.update(epipolar_rooflines(local, fp32_peak, peak_source, args.steps))
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline()
        if args.latency:
            line["config"]["single_fit_latency_ms"] = single_fit_latency(ctx, problems[0], timed)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, record_fields(resident_out))
        print(json.dumps(line))
    ctx.close()
    for c2 in pipe_ctx + pipe_ctx2:
        c2.close()
    if world > 1:
        dist.destroy_process_group()



# ---------------------------------------------------------------------------------------------------------------------
# C5: BASELINE.json configs[4] - ONE homography problem with 1M correspondences (10 % inliers, clustered), NAPSAC over the
# device grid, 10 000 samples; the hypotheses of every round are sharded over the ranks and one NCCL all-gather per round
# exchanges the per-sample scores (strong scaling: the job is fixed, more GPUs finish it sooner). Runs as the second leg of
# the default bench line (`config.c5`, so that the driver's --gpus N runs exercise usac_gpu_nccl_init / ncclAllGather) and
# alone with `--workload c5`.
# ---------------------------------------------------------------------------------------------------------------------
C5_GOLDEN = os.path.join(ROOT, "tests", "golden", "c5_n1_oracle.json")   # the full 10 000-sample fit by the CPU oracle (committed)


def c5_leg(args, rank, world, local, steps, warmup, dump=None):
    """-> dict for config.c5 (every rank returns it; identical on all ranks by construction and asserted so). `dump`: directory
    for rank 0's fit record of the last timed step (--dump-outputs of --workload c5)."""
    import zlib

    import torch

    from ransac_b200 import GpuContext, capi, nccl_unique_id
    from ransac_b200 import dist as D
    from ransac_b200 import generator as gen
    n = args.c5_points
    # samples per round: two rounds cover the 10 000 iterations (5000 + 5000), the same for every rank count - results do not depend on K,
    # samples the sequential loop can no longer reach are neither solved nor scored, and every round costs one exchange
    K = args.c5_round if args.c5_round > 0 else 5000
    pts = gen.make(5, n=n)[0]
    host = torch.from_numpy(pts).pin_memory()
    ctx = GpuContext(local)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    if world > 1:
        ctx.nccl_init(D.broadcast_bytes(nccl_unique_id() if rank == 0 else None), rank, world)
    fit_kw = dict(threshold=THR, confidence=CONF, max_iterations=MAX_IT, seed=1, round_size=K, sampler=capi.SAMPLER_NAPSAC,
                  neighbors=capi.NEIGH_GRID, rank=rank, nranks=world)
    ctx.set_points(capi.EST_HOMOGRAPHY, host)
    ctx.set_neighbors_grid(0, 50)

    def bracket(fn, nsteps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        D.barrier(); torch.cuda.synchronize()
        out = []
        ev0.record(stream)
        for _ in range(nsteps):
            out.append(fn())
        ev1.record(stream)
        D.barrier(); torch.cuda.synchronize()
        return ev0.elapsed_time(ev1), out

    last = [None]

    def step():
        last[0] = ctx.fit_records(**fit_kw)
        r = last[0][0]
        t = ctx.last_timing()
        return (int(r["useful_evals"]), int(r["evals"]), t["launches"], t["score_launches"], t["score_ms"], int(r["iterations"]), int(r["inliers"]),
                int(r["best_hyp"]), zlib.crc32(np.asarray(r["model"], np.float32).tobytes()), int(r["rounds"]))

    def step_e2e():
        ctx.set_points(capi.EST_HOMOGRAPHY, host)          # H2D of the 16 MB point set + the device-side grid build (the reference
        ctx.set_neighbors_grid(0, 50)                       # times its neighbourhood build separately: test/test.cpp:17-29)
        return step()

    # N > 1: first with one NCCL all-gather per round (the hook), then with the exchange over peer memory (IPC windows: the reduce
    # kernel stores into every rank's window over NVLink, select_kernel waits for the flags) - the product's default when attached
    ms_nccl, exchange = None, "none (one GPU)"
    if world > 1:
        bracket(step, warmup)
        ms_nccl_total, st_nccl = bracket(step, steps)
        ms_nccl = D.reduce_max([ms_nccl_total / steps])[0]
        exchange = "NCCL all-gather per round"
        if os.environ.get("USAC_BENCH_EXCHANGE", "peer") != "nccl":
            try:
                ctx.peer_attach(D.allgather_bytes(ctx.peer_export()), rank, world)
                ok = 1.0
            except Exception as e:   # noqa: BLE001
                print(f"bench.py: peer windows unavailable on rank {rank}: {e}", file=sys.stderr)
                ok = 0.0
            all_ok = -D.reduce_max([-ok])[0] >= 1.0
            if not all_ok:
                ctx.peer_detach()                                     # every rank goes back to the NCCL hook
            else:
                exchange = "peer windows over NVLink (stores from the reduce kernel + flags, no collective call)"
    bracket(step, warmup)
    clocks = ClockSampler(local)
    clocks.start()
    ms, st = bracket(step, steps)
    clk = clocks.stop()
    if dump and rank == 0:
        dump_outputs(dump, record_fields(last[0]))
    ms_e2e, st_e2e = bracket(step_e2e, steps)
    t_all = D.reduce_max([ms / steps, ms_e2e / steps])
    sums = D.reduce_sum([sum(x[0] for x in st), sum(x[1] for x in st), sum(x[2] for x in st), sum(x[0] for x in st_e2e) / steps])
    # every rank must hold the same result (the gathered scores and select_kernel are identical everywhere)
    mine = [float(st[-1][5]), float(st[-1][6]), float(st[-1][7]), float(st[-1][8])]
    lo_, hi_ = D.reduce_max(mine), [-v for v in D.reduce_max([-v for v in mine])]
    ranks_agree = lo_ == hi_ == mine
    assert ranks_agree, f"C5: ranks disagree: rank {rank} has {mine}, max {lo_}, min {hi_}"
    parity = None
    if n == 1000000 and os.path.exists(C5_GOLDEN):
        gold = json.load(open(C5_GOLDEN))
        parity = all(int(st[-1][i]) == int(gold[k]) for i, k in ((5, "iterations"), (6, "inliers"), (7, "best_hyp"), (8, "model_crc")))
        assert parity, f"C5: result differs from the single-GPU / oracle record {gold}: {st[-1][5:9]}"
    executed, launches, score_ms = sum(x[1] for x in st), sum(x[3] for x in st), sum(x[4] for x in st)
    info = ctx.device_info()
    peak = 2.0 * 128 * info["sm_count"] * info["sm_clock_khz"] * 1e3 / 1e12
    out = {"workload": f"C5 homography N={n}, 10% inliers (clustered), NAPSAC grid cell 50, max_iter {MAX_IT}, conf {CONF}; one robust fit, "
                       f"hypotheses of every round of {K} samples sharded over {world} GPU(s), one exchange of the per-sample scores per round",
           "scaling": "strong", "steps": steps, "exchange": exchange, "ms_per_fit_nccl": ms_nccl, "ms_per_fit": t_all[0], "evals_per_s": sums[0] / steps / (t_all[0] * 1e-3),
           "evals_executed_per_s": sums[1] / steps / (t_all[0] * 1e-3),
           "iterations": st[-1][5], "inliers": st[-1][6], "best_hyp": st[-1][7], "model_crc": st[-1][8], "rounds": st[-1][9],
           "parity_vs_n1": parity, "parity_note": "iterations / inliers / winning sample / model CRC32 equal tests/golden/c5_n1_oracle.json "
           "(the CPU oracle's full fit, = the 1-GPU result) on every rank", "ranks_agree": bool(ranks_agree),
           "gpu_launches_per_fit": sums[2] / steps / world, "e2e_ms_per_fit": t_all[1], "e2e_evals_per_s": sums[3] / (t_all[1] * 1e-3),
           "h2d_bytes_per_fit": n * 16,
           "score_kernel_frac_of_fp32_peak": 42.0 * executed / (score_ms * 1e-3) / 1e12 / peak, "score_share_of_fit": score_ms / ms,
           "clocks": clk}
    ctx.close()
    return out


def run_c5(args):
    import torch

    from ransac_b200 import dist as D
    local = env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product path has no CPU fallback")
    torch.cuda.set_device(local)
    rank, world = D.init("nccl")
    c5 = c5_leg(args, rank, world, local, args.steps, max(args.warmup, 3), dump=args.dump_outputs)
    if rank == 0:
        line = {"metric": METRIC, "value": c5["evals_per_s"], "unit": "evals/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": c5["ms_per_fit"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": {"workload": c5["workload"], "c5": c5,
                                                "l2": "the 32 MB point set (AoS + pair layout) is L2 resident by design: it is re-read by every model block"},
                "clocks": c5["clocks"], "gpu_launches": int(c5["gpu_launches_per_fit"] * args.steps * world),
                "e2e": {"value": c5["e2e_evals_per_s"], "unit": "evals/s", "h2d_bytes_per_step": c5["h2d_bytes_per_fit"], "d2h_bytes_per_step": 176 + 4 * c5["rounds"],
                        "ms_per_step": c5["e2e_ms_per_fit"], "note": "includes the device-side grid build of set_neighbors_grid"}}
        print(json.dumps(line))
    D.finalize()


def epipolar_rooflines(local, fp32_peak, peak_source, steps=6):
    """roofline_f / roofline_e: the scoring kernel on fundamental (squared Sampson, 33 flop) and essential (symmetric epipolar
    distance, 44 flop) hypotheses: one round of K samples for each of 1184 image pairs of 4000 correspondences with the
    inlier ratios of BASELINE.json's configs 3 and 4 (25 % / 20 %), device resident; CUDA events around the one scoring launch
    of every fit (usac_gpu_last_timing), best of `steps`."""
    from ransac_b200 import GpuContext, capi
    from ransac_b200 import generator as gen
    out = {}
    B = 1184
    # K: the seven-point solver keeps a model for ~15 % of the samples (oriented-epipolar filter), the five-point solver for ~1/3: rounds of
    # 2048 / 1024 samples give ~300 models per image pair - the model count of a 256-sample homography round (the bench's first rounds)
    for name, est, make, thr, flops, K in (("roofline_f", capi.EST_FUNDAMENTAL, lambda s: gen.fundamental(n=N_POINTS, inlier_ratio=0.25, seed=s)[0], 2.0, 33, 2048),
                                           ("roofline_e", capi.EST_ESSENTIAL, lambda s: gen.essential(n=N_POINTS, inlier_ratio=0.2, seed=s)[0], 2.5e-3, 44, 1024)):
        pts = np.concatenate([make(7000 + i) for i in range(B)])
        ctx = GpuContext(local)
        ctx.set_points(est, pts, [N_POINTS] * B)
        best, ev = None, 0.0
        for rep in range(steps + 2):
            res = ctx.fit_records(thr, CONF, K, seed=rep + 1, round_size=K)
            t = ctx.last_timing()
            if rep >= 2 and t["score_launches"] == 1 and (best is None or t["score_ms"] < best):
                best, ev = t["score_ms"], float(res["evals"].sum())
        ctx.close()
        if best:
            ach = flops * ev / (best * 1e-3) / 1e12
            out[name] = {"bound": "fp32", "kernel": f"score_sq_kernel<{'FUNDAMENTAL' if est == capi.EST_FUNDAMENTAL else 'ESSENTIAL'}>", "achieved": ach,
                         "peak": fp32_peak, "unit": "TFLOP/s", "frac": ach / fp32_peak, "flops_per_eval": flops, "evals_per_launch": ev,
                         "launch_ms": best, "steps": steps, "peak_source": peak_source,
                         "workload": f"{B} image pairs x {K} samples x {N_POINTS} correspondences, one scoring launch per fit"}
    return out


def single_fit_latency(ctx, pts, timed):
    """ms per robust fit when ONE image pair is fitted alone (launch/sync latency bound), median of 20."""
    from ransac_b200 import capi
    ctx.set_points(capi.EST_HOMOGRAPHY, pts)
    vals = []
    for i in range(23):
        ms, _ = timed(lambda: ctx.fit(threshold=THR, confidence=CONF, max_iterations=MAX_IT, seed=1), 1)
        if i >= 3:
            vals.append(ms)
    return float(np.median(vals))


def claim_stdout():
    """The contract is ONE JSON line on stdout. Libraries loaded on the way may print there too (NCCL writes its version banner to
    stdout when a communicator is created with NCCL_DEBUG set): file descriptor 1 is pointed at stderr for the whole run and the
    JSON line goes to the real stdout."""
    real = os.fdopen(os.dup(1), "w")
    sys.stdout.flush()
    os.dup2(2, 1)
    sys.stdout = real


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--problems", type=int, default=2368, help="image pairs per GPU and step (2368 = 16 x 148 SMs)")
    ap.add_argument("--ref-problems", type=int, default=256, help="image pairs per step of the CPU reference arm")
    ap.add_argument("--round-size", type=int, default=256, help="samples per round and problem")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--latency", action="store_true", help="also measure the single-fit latency")
    ap.add_argument("--no-epipolar", action="store_true", help="skip the roofline_f / roofline_e legs (Sampson / essential scoring kernels)")
    ap.add_argument("--no-c5", action="store_true", help="skip the second leg (config.c5: the hypothesis-sharded 1M-point fit)")
    ap.add_argument("--pipe", type=int, default=2, help="contexts/streams the e2e arm splits a step over (upload of one part overlaps the fit of another)")
    ap.add_argument("--workload", default="c2", choices=["c2", "c5"], help="c2: batch of independent N=4000 fits (default); c5: one 1M-point fit, hypotheses sharded")
    ap.add_argument("--c5-points", type=int, default=1000000)
    ap.add_argument("--c5-round", type=int, default=0, help="samples per round of the c5 leg (0 = 5000)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the results of the last one (rank 0: one row per "
                    "fit in image-pair order, every field of the fit record) as DIR/<field>.npy, float32 or float64, 64 MB at most. "
                    "The GPU arms fit --problems pairs; the CPU arm (--impl reference) fits max(host cores, --ref-problems) pairs, "
                    "so its dumps from hosts with other core counts agree on the common leading rows only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "native":
        args.warmup = max(args.warmup, 1)
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.workload == "c5":
        run_c5(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
