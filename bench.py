#!/usr/bin/env python
"""Benchmark of the hot path: batched per-object shape-prior GN reconstruction.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2_sdf|cfg2_full|cfg3] [--engine auto|simt|tc]
  python bench.py --impl reference ...      # the CPU restatement of the reference on the host cores

A "step" = one batched call that runs ALL GN iterations of ONE object list (BASELINE config 2 by default:
32 objects x 2048 surface points x 10 iterations, surface-SDF loss, per GPU).  Under torchrun the list has
32 x N objects (N = 8: BASELINE config 4's 256-object batch; weak scaling), every rank builds the same list,
`dsp_slam_b200.distributed.ShardedOptimizer` shards it object-per-GPU (class-sorted contiguous blocks) and
the solved (pose, code, loss, status) records go back to rank 0 INSIDE the step: stored by the solve kernel
straight into rank 0's HBM over NVLink (CUDA-IPC peer mapping; `--exchange nccl` = all-gather instead).
Prints ONE JSON line on rank 0.

  --dump-outputs DIR   after the timed steps, rank 0 writes what the last timed step computed, as the arrays a caller
                       of Optimizer.reconstruct_batch receives (DIR/<name>.npy, float32; NaN where that caller gets
                       None).  The inputs are seeded: the same arguments give the same inputs on every run.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True          # the tree may be read-only: nothing is written into it
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F_FWD = 918_016          # FLOP / row forward   (459,008 MAC; SURVEY.md 8d)
F_BWD = 918_016          # FLOP / row backward-to-input
F_JTJ = 5_254            # FLOP / row J^T J + J^T r

WORKLOADS = {
    # name: (objects/GPU, pts, fg rays, bg rays, class, config, sdf_only, description)
    "cfg2_sdf": (32, 2048, 0, 0, "cars", "config_kitti.json", True,
                 "BASELINE configs[1]: 32 objects x 2048 surface pts x 10 GN iters, surface-SDF loss"),
    "cfg2_full": (32, 2048, 2048, 200, "cars", "config_kitti.json", False,
                  "config 2 full: 32 objects x 2048 pts + 2248 rays x 50 depth samples x 10 GN iters"),
    "slam1": (1, 250, 250, 200, "cars", "config_kitti.json", False,
              "what LocalMapping sends per call (src/LocalMapping_util.cc:179-180): 1 object x 250 LiDAR pts + 450 rays x 50 samples x 10 iters"),
    "cfg3": (8, 256, 64, 18, "chairs", "config_redwood_01053.json", False,
             "BASELINE configs[2]: 8 chairs x 256 pts + 82 rays x 50 samples x 10 iters, initial code"),
    "cfg4": (32, 2048, 0, 0, "cars", "config_kitti.json", True,
             "BASELINE configs[3]: one synthetic car batch of 32 x N objects (256 at 8 GPUs) x 2048 pts x 10 GN iters, "
             "surface-SDF loss, sharded object-per-GPU"),
    "cfg5": (16, 2048, 0, 0, "mixed", "config_kitti.json", True,
             "BASELINE configs[4]: mixed cars+chairs (alternating, two resident decoder weight sets), 16 x N objects "
             "(128 at 8 GPUs) x 2048 pts x 10 GN iters, surface-SDF loss"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2_sdf", choices=list(WORKLOADS))
    ap.add_argument("--engine", default="auto", choices=["auto", "simt", "tc"])
    ap.add_argument("--cpu-sample", type=int, default=4, help="objects in the CPU baseline sample")
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "nccl"],
                    help="multi-GPU result exchange: NVLink peer stores from the solve kernel (default) or NCCL all-gather")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return a


def dump_outputs(out_dir, rec, code_len):
    """(n, RESULT_FLOATS) solver records -> the per-object results a caller of reconstruct_batch receives, stacked."""
    from dsp_slam_b200.distributed import records_to_results
    res = records_to_results(rec, code_len)
    nan = np.float32(np.nan)

    def col(key, shape):
        return np.stack([np.asarray(r[key], np.float32) if r.get(key) is not None else np.full(shape, nan) for r in res])
    arrays = {"t_cam_obj": col("t_cam_obj", (4, 4)), "code": col("code", (code_len,)),
              "is_good": col("is_good", ()), "loss": col("loss", ()), "status": col("status", ()),
              "n_valid": col("n_valid", ()), "n_band": col("n_band", ())}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def make_inputs(workload, world=1):
    """The ONE object list of a step: objects-per-GPU x world detections (identical on every rank)."""
    from dsp_slam_b200 import synth, load_config
    B, M, nfg, nbg, cls, cfgname, sdf_only, _ = WORKLOADS[workload]
    n = B * world
    cfg = load_config(cfgname)
    cfg["optimizer"]["joint_optim"]["num_iterations"] = 10
    clss = [("cars", "chairs")[i & 1] for i in range(n)] if cls == "mixed" else [cls] * n
    objs = synth.make_batch(n, M, nfg if not sdf_only else 0, nbg if not sdf_only else 0, cls=clss,
                            seed0=0, init_code_frac=0.5 if workload == "cfg3" else None)
    ins = []
    for o, c in zip(objs, clss):
        d = dict(t_cam_obj=o["t_cam_obj_init"], pts=o["pts"])
        if not sdf_only:
            d.update(rays=o["rays"], depth=o["depth"])
        if o.get("code_init") is not None:
            d["code"] = o["code_init"]
        if cls == "mixed":
            d["class_id"] = 0 if c == "cars" else 1
        ins.append(d)
    return cfg, ins, clss, sdf_only


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(gpu_index), "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for t, line in self.rows:
            p = [x.strip() for x in line.split(",")]
            if len(p) < 7:
                continue
            try:
                if t0 - 0.05 <= t <= t1 + 0.15:
                    sm.append(float(p[0]))
                smax = float(p[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active") and t0 - 0.05 <= t <= t1 + 0.15:
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_baseline(workload, n_sample, steps=1, warmup=0):
    """The numpy restatement of the reference (oracle/dsp_oracle.py) on the host cores: objects one per
    call in a Python loop, exactly how the reference batches (src/LocalMapping_util.cc:165-203)."""
    from oracle import dsp_oracle as O
    cfg, ins, clss, sdf_only = make_inputs(workload, 1)
    dws = {c: O.DecoderWeights.from_npz(os.path.join(ROOT, "tests", "golden", f"decoder_{c}.npz")) for c in set(clss)}
    dw = dws[clss[0]]
    ocfg = O.GNConfig.from_json_dict(cfg)
    sample = list(zip(ins[:n_sample], clss[:n_sample]))

    def one_pass():
        for o, c in sample:
            O.reconstruct_object(dws[c], ocfg, o["t_cam_obj"], o["pts"], o.get("rays"), o.get("depth"),
                                 code=o.get("code"), sdf_only=sdf_only)
    # always one untimed object first: BLAS thread pool spin-up / page-in are not the steady state
    o = sample[0][0]
    O.reconstruct_object(dw, ocfg, o["t_cam_obj"], o["pts"], o.get("rays"), o.get("depth"), code=o.get("code"), sdf_only=sdf_only)
    # give the CPU leg its best thread count: these GEMMs are small (2048x256x256) and OpenBLAS with one
    # thread per core of a 100+-core host is slower than with 8-32 threads
    global _CPU_THREADS
    try:
        from threadpoolctl import threadpool_limits
        x = np.concatenate([np.zeros((o["pts"].shape[0], 64), np.float32), np.asarray(o["pts"], np.float32)], 1)
        best, cands = None, sorted({t for t in (4, 8, 16, 32, 64, os.cpu_count()) if t <= os.cpu_count()})
        for t in cands:
            with threadpool_limits(limits=t):
                O.decoder_value_and_input_grad(dw, x)
                t0 = time.perf_counter()
                for _ in range(3):
                    O.decoder_value_and_input_grad(dw, x)
                dt = time.perf_counter() - t0
            if best is None or dt < best[1]:
                best = (t, dt)
        _CPU_THREADS = best[0]
        threadpool_limits(limits=_CPU_THREADS)
    except Exception:
        _CPU_THREADS = os.cpu_count()
    for _ in range(warmup):
        one_pass()
    t0 = time.perf_counter()
    for _ in range(steps):
        one_pass()
    dt = (time.perf_counter() - t0) / steps
    return len(sample) / dt, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B, M, nfg, nbg, cls, cfgname, sdf_only, desc = WORKLOADS[args.workload]
    steps = args.steps
    val, dt = cpu_baseline(args.workload, args.cpu_sample, steps=steps, warmup=min(args.warmup, 1))
    cores = os.cpu_count()
    out = {
        "impl": "reference", "metric": "object-recons/sec (2048 pts, 10 GN iters)", "value": val, "unit": "objects/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": min(args.warmup, 1), "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "objects_per_step": args.cpu_sample},
        "cpu_baseline": {"value": val, "unit": "objects/s", "cores": _CPU_THREADS or cores, "kind": "port",
                         "host_cores": cores, "cpu_model": cpu_model(),
                         "sample": f"{args.cpu_sample} of the {B} objects per step, numpy/OpenBLAS fp32 restatement "
                                   f"(oracle/dsp_oracle.py), one object per call like the reference; thread count = the "
                                   f"fastest of 4..{cores} for these 2048x256x256 GEMMs"},
        "e2e": {"value": val, "unit": "objects/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


_CPU_THREADS = None


class _CudaArray:
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (ptr, False), "version": 3}


def run_ours(args):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as g
    g.build()
    from dsp_slam_b200.optimizer import Optimizer
    from dsp_slam_b200.distributed import ShardedOptimizer
    from dsp_slam_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    B, M, nfg, nbg, cls, cfgname, sdf_only, desc = WORKLOADS[args.workload]
    n_total = B * world
    cfg, ins, clss, sdf_only = make_inputs(args.workload, world)          # ONE list, identical on every rank
    G = os.path.join(ROOT, "tests", "golden")
    decs = [os.path.join(G, "decoder_cars.npz"), os.path.join(G, "decoder_chairs.npz")] if cls == "mixed" \
        else [os.path.join(G, f"decoder_{cls}.npz")]
    opt = Optimizer(decs[0], cfg, device=local, engine=None if args.engine == "auto" else args.engine, sdf_only=sdf_only,
                    extra_decoders=decs[1:])
    solver = opt.solver
    stream = torch.cuda.current_stream()
    solver.set_stream(stream.cuda_stream)
    engine = {1: "simt-fp32", 2: "tcgen05-3xf16"}[solver.engine]
    sh = ShardedOptimizer(opt, exchange=args.exchange) if world > 1 else None
    exchange = sh.exchange if sh else "none (single GPU)"

    # ---- device-timed: the shard is resident in HBM before the timed region ---------------------------------
    if sh:
        sh.upload_shard(ins)
        n_mine = len(sh._idx)
    else:
        solver.upload(ins)
        n_mine = n_total
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step():
        if sh is None:
            solver.run(0)
        else:
            sh.run_shard(0)                 # peer: records stored into rank 0's HBM + flag; rank 0 waits for all flags
            if sh.exchange == "nccl":
                sh.exchange_async_nccl()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_loop(fn, steps):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        t0 = time.perf_counter()
        for a, b in ev:
            flush.fill_(1)                  # L2 flush (256 MiB write) outside the event pair
            a.record(stream)
            fn()
            b.record(stream)
        barrier()
        t1 = time.perf_counter()
        return sum(a.elapsed_time(b) for a, b in ev) / steps, t0, t1

    def max_over_ranks(x, op=None):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=op or dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local) if rank == 0 else None      # started before the warm-up: nvidia-smi takes ~0.2 s to deliver its first sample
    for _ in range(max(args.warmup, 3)):
        step()
    if sampler is not None:
        t_wait = time.perf_counter()
        while not sampler.rows and time.perf_counter() - t_wait < 2.0:
            time.sleep(0.02)
    ms_local, t0, t1 = timed_loop(step, args.steps)
    clocks = sampler.stop(t0, t1) if sampler else None
    if args.dump_outputs:               # before anything else runs on the resident batch
        rec = sh.gather_records() if sh else np.frombuffer(solver.results_raw(), np.float32).reshape(n_total, -1)
        if rank == 0:
            dump_outputs(args.dump_outputs, rec, opt.code_len)
    launches_per_step = solver.counters()["kernel_launches"]
    ms = max_over_ranks(ms_local)
    value = n_total / (ms * 1e-3)

    # per-rank split of the step (root cause of any scaling loss): the solver's own kernels vs the exchange
    kernel_ms_local = solver.counters()["total_ms"]                 # CUDA events around the last run's kernels
    multi = None
    if world > 1:
        wait_ms = sh.peer.wait_ms() if (sh.peer is not None and rank == 0) else 0.0
        ms_noex, _, _ = timed_loop(lambda: solver.run(0), max(3, min(args.steps, 10)))    # same shard, no exchange
        multi = {
            "exchange": ("NVLink peer stores from the solve kernel into rank 0's HBM (CUDA IPC), per-rank flag, no "
                         "collective kernel") if sh.exchange == "peer" else "NCCL all_gather_into_tensor on the solver stream",
            "step_ms_per_rank": {"max": ms, "min": -max_over_ranks(-ms_local)},
            "kernel_ms_per_rank": {"max": max_over_ranks(kernel_ms_local), "min": -max_over_ranks(-kernel_ms_local)},
            "ms_per_step_without_exchange": max_over_ranks(ms_noex),
            "root_wait_ms_last_step": wait_ms,
            "objects_total": n_total, "objects_this_rank": n_mine,
        }
        if sh.peer is not None:
            sh.upload_shard(ins)            # re-bind after the plain runs (same resident shard)

    # correctness of what was timed: every object of the whole list converged (rank 0 holds all records)
    if sh:
        sh.run_shard(0)
        rec = sh.gather_records()
        n_good = int((rec.view(np.int32)[:, 81] == 0).sum()) if rec is not None else -1
    else:
        out = solver.results_raw()
        n_good = sum(1 for i in range(n_total) if out[i].status == 0)

    # ---- end to end through the public call: host buffers, pack + H2D + all iterations + exchange + D2H ------
    def e2e_call():
        return sh.reconstruct_batch(ins) if sh else opt.reconstruct_batch(ins)
    for _ in range(2):
        e2e_call()
    barrier()
    e2e_steps = max(3, min(args.steps, 10))
    te = time.perf_counter()
    for _ in range(e2e_steps):
        res = e2e_call()
    torch.cuda.synchronize()
    e2e_ms = max_over_ranks((time.perf_counter() - te) / e2e_steps * 1e3)
    if rank == 0:
        assert len(res) == n_total and sum(1 for r in res if r.is_good) == n_good, "e2e results incomplete"
    h2d = sum(o["pts"].nbytes + 64 + 256 + 40 + (o["rays"].nbytes + o["depth"].nbytes if "rays" in o else 0) for o in ins)
    d2h = n_total * 4 * _lib.RESULT_FLOATS

    # ---- roofline of the dominant kernel (decoder fwd+bwd+JtJ over this rank's rows), live CUDA events -------
    if sh:
        sh.upload_shard(ins)
    else:
        solver.upload(ins)
    solver.enable_timing(True)
    dec_ms = []
    for _ in range(3):
        solver.run(0)
        solver.results_raw()
        c = solver.counters()
        dec_ms.append(c["decoder_ms"])
        solve_ms = c["solve_ms"]; total_ms = c["total_ms"]
    solver.enable_timing(False)
    c = solver.counters()
    iters = 10
    persistent = c["kernel_launches"] <= 3
    n_dec_launch = 1 if persistent else iters * (1 if sdf_only else 3)
    rows_fb, rows_f = c["rows_fwd_bwd"], c["rows_fwd_only"]
    flop_alg = rows_fb * (F_FWD + F_BWD + F_JTJ) + rows_f * F_FWD
    dec_ms_med = float(np.median(dec_ms))
    achieved = flop_alg / (dec_ms_med * 1e-3) / 1e12
    peaks, peak_src = None, "fallback (B200_PROFILING.md)"
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak, peak_sus = 1590.0, 1400.0
    if os.path.isfile(pk):
        peaks = json.load(open(pk))
        peak = float(peaks.get("bf16_tflops", peak))
        peak_sus = float(peaks.get("bf16_tflops_sustained", peak_sus))
        peak_src = "MEASURED_PEAKS.json bf16_tflops (burst figure: the kernel lasts ~3 ms); frac_of_sustained uses bf16_tflops_sustained"
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(tp):
        traffic = json.load(open(tp)).get(f"{args.workload}:{engine}")

    if rank == 0:
        cpu_val, cpu_dt = cpu_baseline(args.workload, args.cpu_sample)
        sched = "persistent object-pipelined kernel (device work queue)" if persistent else "one launch per term per iteration"
        out = {
            "metric": "object-recons/sec (2048 pts, 10 GN iters)", "value": value, "unit": "objects/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if solver.engine == 1 else "f16x3-split (fp32 accumulate)", "data": "synthetic",
            "config": {"workload": desc, "objects_per_gpu": B, "objects_per_step": n_total, "points": M, "gn_iterations": 10,
                       "engine": engine,
                       "parallelism": f"one {n_total}-object list sharded object-per-GPU x{world} (class-sorted contiguous blocks); "
                                      f"results to rank 0 in original order; exchange: {exchange}",
                       "schedule": sched,
                       "l2": "flushed between timed steps (256 MiB write, outside the event pairs)",
                       "decoder": "DeepSDF 8x256, L=64, latent_in=[4] (fitted fixture weights)",
                       "good_objects": f"{n_good}/{n_total}"},
            "e2e": {"value": n_total / (e2e_ms * 1e-3), "unit": "objects/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms,
                    "path": ("ShardedOptimizer.reconstruct_batch(one list): pack + H2D of every rank's shard, all GN iterations, "
                             "records to rank 0, D2H + unpack on rank 0") if sh else "Optimizer.reconstruct_batch (pack + H2D + run + D2H + unpack)"},
            "gpu_launches": int(launches_per_step * args.steps),
            "clocks": clocks,
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak, "frac_of_sustained": achieved / peak_sus, "traffic": traffic, "peak_source": peak_src,
                         "note": "achieved counts 1x algorithmic FLOPs; the tensor pipe issues 3x (split-fp16 passes)",
                         "kernel": ("k_gn_persistent: all GN iterations of all objects in one launch (decoder tiles + "
                                    "in-kernel scans and solves, " + engine + ")") if persistent else "decoder fwd+bwd+JtJ (" + engine + ")",
                         "alg_flop_per_run": flop_alg, "decoder_ms_per_run": dec_ms_med,
                         "solve_ms_per_run": solve_ms, "run_ms_with_event_overhead": total_ms,
                         "decoder_launches_per_run": n_dec_launch},
            "cpu_baseline": {"value": cpu_val, "unit": "objects/s", "cores": _CPU_THREADS or os.cpu_count(), "kind": "port",
                             "host_cores": os.cpu_count(), "cpu_model": cpu_model(),
                             "sample": f"{args.cpu_sample} of the {n_total} objects, numpy/OpenBLAS fp32 restatement of the "
                                       f"reference (oracle/dsp_oracle.py), one object per call"},
        }
        if multi:
            out["multi_gpu"] = multi
        print(json.dumps(out), flush=True)
    if sh:
        barrier()
        sh.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
