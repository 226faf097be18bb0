#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json metric) on N GPUs of one node.

A "step" = one pass of the hot path over one batch of synthetic OCP instances: a cold Controller::step for every
instance of the workload.  Default workload = BASELINE configs[1] (batch 1024 per GPU, unicycle quadratic-form, N=50,
5 circular obstacles); `--config 3|4|5` measures BASELINE configs[2..4] through the same code.

  python bench.py --gpus 1 --steps K --warmup W                       (single GPU)
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...   (one rank per GPU)
  python bench.py --impl reference ...                                (CPU arm: the oracle port on the host cores)

Rank 0 prints ONE JSON line.
  value        whole-job converged solves/s, inputs already resident in HBM (mpcb200_solve_resident: ONE launch of the
               persistent solve kernel per step, L2 flushed between steps, CUDA events on the work stream, max over ranks)
  e2e          the same metric through mpcb200_step_batch with pinned HOST buffers (H2D + D2H inside the timed region)
  roofline     the KKT factorisation kernel (kkt_warp_kernel): algorithmic bytes of SURVEY 8(d) x the instances of a launch
               / its CUDA-event time, timed alone inside this run on the records of the batch, against the measured HBM peak
  cpu_baseline the CPU oracle (plain-C port of the algorithm, test infrastructure) on a bounded sample of the workload
  configs      driver-visible numbers for the other BASELINE configurations (cfg 3 and the horizon sweep at N=1 GPU;
               cfg 4 = 16 384 via-point instances split over the ranks of this run: strong scaling over the driver's runs)

--dump-outputs DIR writes what the last timed step returned (on rank 0: instances [0, batch)) as DIR/<name>.npy, float64:
u_seq [B, N, 2], x_seq [B, N, 3], dt, status, kkt_err, iters [B] and instance [B] (the instance index of each row).  Above
64 MB in all, the rows are a fixed seeded sample.  The inputs are seeded, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

UNIT = "solves/s"
WORKLOADS = {
    2: ("converged MPC solves/sec (N=50 unicycle quadratic-form OCP, 5 obstacles, batched)", 1024,
        "BASELINE configs[1]: batch=1024 per GPU, unicycle quadratic_form, N=50, fixed dt=0.3, 5 circular obstacles, "
        "rate limits 0.2, tol 1e-6, max_iter 100, cold start"),
    3: ("converged MPC solves/sec (N=80 carlike minimum-time OCP, polygon footprint, batched)", 4096,
        "BASELINE configs[2]: batch=4096 per GPU, simple_car (rear drive, L=0.4) minimum_time, N=80, free dt, polygon "
        "footprint (9 vertices), 5 point/circle obstacles, tol 1e-6, max_iter 100, cold start"),
    4: ("converged MPC solves/sec (N=50 unicycle quadratic-form OCP with via-points, batched)", 2048,
        "BASELINE configs[3]: batch=2048 per GPU (16384 over 8), unicycle quadratic_form + via-point attraction, N=50, "
        "5 circular obstacles, 2 via-points, tol 1e-6, max_iter 100, cold start"),
    5: ("converged MPC solves/sec (unicycle quadratic-form OCP, horizon N, batched)", 2048,
        "BASELINE configs[4]: batch=2048, unicycle quadratic_form, horizon N in {20,50,100,200}, 5 circular obstacles"),
}


def kkt_bytes_per_instance(cfg):
    """SURVEY 8(d): w * ((46 + 4*[rate limits] + 3*[dt free]) * (N-1) + 12) bytes, fp64."""
    rate = any(cfg.du_ub[i] < 1e29 or cfg.du_lb[i] > -1e29 for i in range(2))
    words = 46 + (4 if rate else 0) + (3 if cfg.variable_dt else 0)
    return 8 * (words * (cfg.n - 1) + 12)


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst: kernel timed alone)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def host_cores():
    """Threads this process may really use: the affinity mask, capped by the cgroup CPU quota (cpu.max)."""
    try:
        n_aff = len(os.sched_getaffinity(0))
    except Exception:
        n_aff = os.cpu_count() or 1
    quota = None
    for p in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(p).read().split()
            if p.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:
            continue
    n = n_aff
    if quota is not None:
        n = max(1, min(n_aff, int(quota + 0.5)))
    return n, {"os_cpu_count": os.cpu_count(), "affinity": n_aff, "cgroup_quota": quota}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = False
        self.rows = []

    def run(self):
        try:
            self._run_nvml()
        except Exception:
            self._run_smi()

    def _run_nvml(self):
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        bits = [("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4)]
        while not self.stop_flag:
            sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
            except Exception:
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            try:
                pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
            except Exception:
                pw = 0.0
            self.rows.append([str(sm), str(mx), str(pw)] + ["Active" if (r & b) else "Not Active" for _, b in bits])
            time.sleep(0.01)

    def _run_smi(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                o = subprocess.check_output(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                             "-i", str(self.index)], timeout=5).decode().strip()
                self.rows.append([c.strip() for c in o.split(",")])
            except Exception:
                pass
            time.sleep(0.03)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, res):
    """The arrays of one step's result dict as out_dir/<name>.npy (float64); rows sampled with a fixed seed above 64 MB."""
    names = ("u_seq", "x_seq", "dt", "status", "kkt_err", "iters")
    B = res["status"].shape[0]
    row_bytes = 8 * (1 + sum(res[k][0].size for k in names))   # + the instance index
    rows = np.arange(B)
    budget = DUMP_LIMIT_BYTES - 4096   # room for the .npy headers
    if B * row_bytes > budget:
        rows = np.sort(np.random.default_rng(0).choice(B, budget // row_bytes, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "instance.npy"), rows.astype(np.float64))
    for k in names:
        np.save(os.path.join(out_dir, k + ".npy"), np.asarray(res[k][rows], dtype=np.float64))


def cpu_arm(cfg, data_fn, seconds_target, threads):
    """The CPU oracle (port) on a bounded sample of the same workload, on the host threads this process may use."""
    from oracle import oracle_py as orc
    n = max(threads * 8, 32)
    data = data_fn(n)
    t = time.time()
    out = orc.step_batch(cfg, data, n_threads=threads)
    el = time.time() - t
    if el < seconds_target / 4:   # grow the sample towards the time target (bounded)
        n2 = int(min(n * (seconds_target / 2) / max(el, 1e-3), 32768))
        data = data_fn(n2)
        t = time.time()
        out = orc.step_batch(cfg, data, n_threads=threads)
        el = time.time() - t
        n = n2
    conv = int((out["status"] == 0).sum())
    return conv / el, n, conv, el


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5], help="BASELINE configuration (SURVEY 8d numbering)")
    ap.add_argument("--horizon", type=int, default=50, help="grid points N for --config 5")
    ap.add_argument("--batch", type=int, default=0, help="instances per GPU (default: the configuration's batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-configs", action="store_true", help="skip the secondary blocks (cfg 3 / 4 / horizon sweep / queue)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    from mpc_local_planner_b200 import capi, configs
    cid = args.config
    metric, default_batch, workload = WORKLOADS[cid]
    n_h = args.horizon if cid == 5 else None
    cfg = configs.config_for(cid, n=n_h, tol=1e-6)
    B = args.batch or default_batch
    threads, cores_info = host_cores()

    # ------------------------------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        from oracle import oracle_py as orc
        sample = max(threads * 32, 256)
        data = configs.generate(cid, sample, n=n_h)
        for _ in range(max(args.warmup, 0)):
            orc.step_batch(cfg, data, n_threads=threads)
        t0 = time.time()
        conv = 0
        for _ in range(args.steps):
            out = orc.step_batch(cfg, data, n_threads=threads)
            conv += int((out["status"] == 0).sum())
        el = time.time() - t0
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, out)
        val = conv / el
        print(json.dumps({
            "impl": "reference", "metric": metric, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": el / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload},
            "note": "reference arm = CPU oracle port of the same algorithm (the reference's control_box_rst + Ipopt stack cannot "
                    "be built here: no ROS/Eigen/Ipopt, see DESIGN.md)",
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "cores_detail": cores_info, "kind": "port",
                             "sample": f"{sample} instances of the workload per step, {args.steps} steps"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return 0

    # ------------------------------------------------------------------------------------------ our arm
    import torch
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the solver has no CPU fallback"}))
        return 1
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = local_rank if world > 1 else 0
    torch.cuda.set_device(dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max_sum(tmax, tsum):
        """(max over ranks of tmax, sum over ranks of tsum); every rank calls it the same number of times"""
        if dist is None:
            return list(tmax), list(tsum)
        a = torch.tensor(list(tmax), dtype=torch.float64, device=f"cuda:{dev}")
        b = torch.tensor(list(tsum), dtype=torch.float64, device=f"cuda:{dev}")
        dist.all_reduce(a, op=dist.ReduceOp.MAX)
        dist.all_reduce(b, op=dist.ReduceOp.SUM)
        return [float(x) for x in a], [float(x) for x in b]

    stream = torch.cuda.Stream(device=dev)

    def pinned(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return t.numpy(), t

    def measure(cid_, cfg_, B_, steps, warmup, first, want_e2e, want_gather, order_by_history=1):
        """K timed cold batch solves of one workload on this rank.  Returns a dict of local results."""
        data = configs.generate(cid_, B_, first=first, n=cfg_.n if cid_ == 5 else None)
        solver = capi.BatchSolver(cfg_, B_, device=dev)
        solver.set_stream(stream.cuda_stream)
        solver.set_option(capi.OPT_ORDER_BY_HISTORY, order_by_history)
        N = cfg_.n
        send = torch.empty(B_ * (N - 1) * 2, dtype=torch.float64, device=f"cuda:{dev}")
        recv = torch.empty(world * B_ * (N - 1) * 2, dtype=torch.float64, device=f"cuda:{dev}") if (world > 1 and want_gather) else None
        # The all-gather of step i runs beside the solve of step i+1 (async NCCL work; the work stream waits for it only before
        # the send buffer is written again and at the end of the timed region), so the ranks are not re-synchronised every step.
        gather = {"work": None}

        def gather_wait():
            if gather["work"] is not None:
                gather["work"].wait()
                gather["work"] = None

        def gather_controls():
            if recv is not None:
                gather_wait()
                solver.export_controls(send.data_ptr())
                gather["work"] = dist.all_gather_into_tensor(recv, send, async_op=True)

        def resident_step():
            solver.flush_l2()   # the working set of a batch fits in the 126 MB L2: evict between steps
            solver.solve_resident(cold=True)
            gather_controls()

        def timed(fn, n):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            with torch.cuda.stream(stream):
                e0.record(stream)
                last = None
                for _ in range(n):
                    last = fn()
                gather_wait()
                e1.record(stream)
            barrier()
            return e0.elapsed_time(e1) * 1e-3, last

        solver.upload(data["x0"], data["xf"], data["u_prev"], data["u_prev_dt"], data["obstacles"], data["viapoints"])
        with torch.cuda.stream(stream):
            for _ in range(warmup):
                resident_step()
        torch.cuda.synchronize()
        solver.stats_reset()
        sampler = ClockSampler(dev)
        sampler.start()
        el, _ = timed(resident_step, steps)
        sampler.stop_flag = True
        st = solver.stats()
        res = solver.fetch()
        out = {"el": el, "res": res, "conv": int((res["status"] == 0).sum()), "iters_mean": float(res["iters"].mean()), "stats": st,
               "clocks": sampler.summary(), "solver": solver, "data": data, "timed": timed, "gather_controls": gather_controls}
        if want_e2e:
            keep = []
            hin = {}
            for k_ in ("x0", "xf", "u_prev"):
                hin[k_], t_ = pinned(data[k_]); keep.append(t_)
            ob = vp = None
            if data["obstacles"] is not None:
                ob = []
                for a in data["obstacles"]:
                    h_, t_ = pinned(a); ob.append(h_); keep.append(t_)
                ob = tuple(ob)
            if data["viapoints"] is not None:
                vp = []
                for a in data["viapoints"]:
                    h_, t_ = pinned(a); vp.append(h_); keep.append(t_)
                vp = tuple(vp)
            hout = solver.alloc_outputs(B_, pin=lambda a: pinned(a))   # pinned result buffers, reused by every step

            def e2e_step():
                solver.reset()
                solver.flush_l2()
                o = solver.step(hin["x0"], hin["xf"], hin["u_prev"], data["u_prev_dt"], ob, vp, out=hout)  # H2D, solve, D2H
                gather_controls()
                return o
            with torch.cuda.stream(stream):
                for _ in range(2):
                    e2e_step()
            torch.cuda.synchronize()
            st0 = solver.stats()
            e2e_steps = max(3, steps // 2)
            el_e2e, o = timed(e2e_step, e2e_steps)
            st1 = solver.stats()
            out.update(el_e2e=el_e2e, e2e_steps=e2e_steps, conv_e2e=int((o["status"] == 0).sum()),
                       h2d=(st1["h2d_bytes"] - st0["h2d_bytes"]) // e2e_steps, d2h=(st1["d2h_bytes"] - st0["d2h_bytes"]) // e2e_steps,
                       keep=keep)
        return out

    # ================= the contract workload =================
    m = measure(cid, cfg, B, args.steps, args.warmup, rank * B, True, True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, m["res"])
    (el, el_e2e), (conv_total, conv_e2e_total) = reduce_max_sum([m["el"], m["el_e2e"]], [m["conv"], m["conv_e2e"]])
    solver, st, N = m["solver"], m["stats"], cfg.n

    # ---- roofline: the KKT kernel alone on the first-iteration records of this batch (every instance live), L2 flushed
    #      between the launches, CUDA events on the work stream around each launch ----
    peak, peak_src = hbm_peak()
    bpi = kkt_bytes_per_instance(cfg)
    solver.reset()
    solver.set_option(capi.OPT_SOLVE_MODE, capi.SOLVE_PHASED)
    solver.run_phase(capi.PHASE_INIT); solver.run_phase(capi.PHASE_ASSOCIATE); solver.run_phase(capi.PHASE_EVAL)
    solver.stats_reset()
    kkt_ms = solver.time_phase(capi.PHASE_KKT, reps=20, flush_l2=True)
    stk = solver.stats()
    sweeps = stk["kkt_sweeps"] / max(stk["kkt_instances"], 1)
    solver.set_option(capi.OPT_SOLVE_MODE, capi.SOLVE_FUSED)
    achieved = B * bpi / (kkt_ms * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "kkt_traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            if tj.get("batch") == B and tj.get("config") == cid:
                traffic = int(tj["dram_bytes_per_launch"])   # ncu --set full on this kernel at this batch (cold caches)
        except Exception:
            traffic = None
    # share of the solve the KKT phase takes (SM cycles counted by the persistent kernel itself)
    ph = st["ms"]
    ph_sum = sum(ph) if sum(ph) > 0 else 1.0
    roofline = {"bound": "hbm", "kernel": "kkt_warp_kernel (warp-cooperative Riccati factorisation + solve, one warp per instance)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_instance": bpi, "instances_per_launch": B, "avg_launch_ms": kkt_ms,
                "sweeps_per_instance": sweeps,
                "how": "kernel timed alone in this run: 20 launches on the batch's first-iteration records, L2 flushed before each, "
                       "CUDA events on the launching stream",
                "in_solve": {"kkt_share_of_cta_time": ph[capi.PHASE_KKT] / ph_sum,
                             "kkt_calls": st["kkt_instances"], "sweeps_per_call": st["kkt_sweeps"] / max(st["kkt_instances"], 1),
                             "algorithmic_gbs_over_the_step": st["kkt_instances"] * bpi / el / 1e9,
                             "note": "inside the persistent solve kernel the records never leave shared memory"},
                "dominant_kernel": {"kernel": "solve_fused_kernel (one launch = one step: every instance from the initial guess to convergence)",
                                    "share_of_step": 0.94, "share_source": "profiles/r2_launch_shares.txt (ncu launch list of this command)",
                                    "avg_launch_ms": el / args.steps * 1e3,
                                    "algorithmic_gbs": st["kkt_instances"] * bpi / el / 1e9, "frac_of_hbm_peak": st["kkt_instances"] * bpi / el / 1e9 / peak,
                                    "dram_bytes_per_launch_ncu": 43140864,
                                    "note": "SURVEY 8d's per-unit bytes (the KKT records and steps of every instance-iteration) x the "
                                            "instance-iterations of a step / the step time.  The kernel keeps those records in shared memory "
                                            "(ncu: 7.9 MB read + 35.2 MB written per launch, profiles/r2_fused_ncu.txt), so it is nowhere near "
                                            "the HBM roofline by construction: it is bound by the latency of one interior-point iteration "
                                            "(DESIGN.md 4).  The stand-alone KKT kernel above is the one kernel of the path that streams its "
                                            "data through HBM, hence the roofline kernel."}}

    # ================= secondary blocks =================
    extra = {}
    err_flag = 0.0
    if not args.no_extra_configs:
        # (a) the K steps' instances as ONE queue through the persistent kernel (mpcb200_solve_stream), host buffers in and out
        try:
            reps = min(args.steps, 16)
            data = m["data"]
            tile = lambda a: np.ascontiguousarray(np.concatenate([a] * reps))
            q = dict(x0=tile(data["x0"]), xf=tile(data["xf"]), u_prev=tile(data["u_prev"]),
                     obstacles=tuple(tile(a) for a in data["obstacles"]) if data["obstacles"] is not None else None,
                     viapoints=tuple(tile(a) for a in data["viapoints"]) if data["viapoints"] is not None else None)
            with torch.cuda.stream(stream):
                solver.solve_stream(q["x0"], q["xf"], q["u_prev"], data["u_prev_dt"], q["obstacles"], q["viapoints"])
            torch.cuda.synchronize()
            el_q, sout = m["timed"](lambda: solver.solve_stream(q["x0"], q["xf"], q["u_prev"], data["u_prev_dt"], q["obstacles"], q["viapoints"]), 1)
            extra["_queue"] = (el_q, int((sout["status"] == 0).sum()), reps)
        except Exception as e:   # never take the contract line down; the collectives below still run on every rank
            extra["_queue"] = (1.0, 0, 0)
            extra["queue_error"] = repr(e)
            err_flag = 1.0
    solver.close()
    if not args.no_extra_configs:
        (elq,), (convq,) = reduce_max_sum([extra["_queue"][0]], [extra["_queue"][1]])
        reps = extra.pop("_queue")[2]
        if reps:
            extra["queue"] = {"value": convq / elq, "unit": UNIT, "instances_per_gpu": reps * B, "ms_per_batch": elq / reps * 1e3,
                              "what": "the same instances as ONE queue of K x batch through the persistent kernel (mpcb200_solve_stream: "
                                      "continuous batching), host buffers in and out; results are bit-identical to the batch solves"}
        # (b) BASELINE configs[3]: 16 384 via-point instances split over the ranks of this run (strong scaling across runs)
        try:
            g = 16384
            b4 = g // world
            c4 = configs.config_for(4, tol=1e-6)
            m4 = measure(4, c4, b4, 3, 3, rank * b4, False, True)
            r4 = (m4["el"], m4["conv"])
            m4["solver"].close()
        except Exception as e:
            r4 = (1.0, 0)
            extra["cfg4_error"] = repr(e)
        (el4,), (conv4,) = reduce_max_sum([r4[0]], [r4[1]])
        extra["cfg4_global16384"] = {"value": conv4 * 3 / el4, "unit": UNIT, "global_batch": 16384, "batch_per_gpu": 16384 // world,
                                     "ms_per_step": el4 / 3 * 1e3, "scaling": "strong", "converged_fraction": conv4 / 16384.0,
                                     "workload": WORKLOADS[4][2]}
        if world == 1 and cid == 2:
            # (c) the cold start exactly as the reference builds it (config.reference_initial_guess = 1: straight line, zero
            #     controls, no solver-side preprocessing), same instances: how many converge within the 100 iterations, how fast
            try:
                cr = configs.config_for(2, tol=1e-6)
                cr.reference_initial_guess = 1
                mr = measure(2, cr, B, 5, 3, 0, False, False)
                extra["reference_initial_guess"] = {"value": mr["conv"] * 5 / mr["el"], "unit": UNIT, "ms_per_step": mr["el"] / 5 * 1e3,
                                                    "converged_fraction": mr["conv"] / float(B), "mean_ipm_iterations": mr["iters_mean"],
                                                    "what": "config.reference_initial_guess = 1 (the reference's initial guess, "
                                                            "full_discretization_grid_base_se2.cpp:192-239); the headline uses the default 0 "
                                                            "(bumped-line choice + repair of violated obstacle rows, DESIGN.md)"}
                mr["solver"].close()
            except Exception as e:
                extra["reference_guess_error"] = repr(e)
            # (c2) the headline workload with the queue in index order (MPCB200_OPT_ORDER_BY_HISTORY = 0): every step of this bench solves
            #      the SAME instances, so the default order -- longest first by the previous solve's iteration counts of the same slots --
            #      is an exact hint here; in a fleet it is as good as a robot's difficulty persists from cycle to cycle
            try:
                mo = measure(2, configs.config_for(2, tol=1e-6), B, 10, 3, 0, False, False, order_by_history=0)
                extra["index_order"] = {"value": mo["conv"] * 10 / mo["el"], "unit": UNIT, "ms_per_step": mo["el"] / 10 * 1e3,
                                        "what": "same workload, queue in index order (no history)"}
                mo["solver"].close()
            except Exception as e:
                extra["index_order_error"] = repr(e)
            # (d) BASELINE configs[2] and the horizon sweep of configs[4], one GPU
            try:
                c3 = configs.config_for(3, tol=1e-6)
                m3 = measure(3, c3, 4096, 3, 3, 0, False, False)
                extra["cfg3_b4096"] = {"value": m3["conv"] * 3 / m3["el"], "unit": UNIT, "ms_per_step": m3["el"] / 3 * 1e3,
                                       "converged_fraction": m3["conv"] / 4096.0, "workload": WORKLOADS[3][2]}
                m3["solver"].close()
                sweep = []
                for n_ in (20, 50, 100, 200):
                    c5 = configs.config_for(5, n=n_, tol=1e-6)
                    d5 = configs.generate(5, 2048, n=n_)
                    s5 = capi.BatchSolver(c5, 2048, device=dev)
                    s5.set_stream(stream.cuda_stream)
                    s5.upload(d5["x0"], d5["xf"], d5["u_prev"], d5["u_prev_dt"], d5["obstacles"], d5["viapoints"])
                    s5.set_option(capi.OPT_SOLVE_MODE, capi.SOLVE_PHASED)
                    s5.run_phase(capi.PHASE_INIT); s5.run_phase(capi.PHASE_ASSOCIATE); s5.run_phase(capi.PHASE_EVAL)
                    ms5 = s5.time_phase(capi.PHASE_KKT, reps=10, flush_l2=True)
                    s5.set_option(capi.OPT_SOLVE_MODE, capi.SOLVE_FUSED)
                    s5.flush_l2()
                    t5 = s5.solve_resident(cold=True)
                    o5 = s5.fetch()
                    gbs = 2048 * kkt_bytes_per_instance(c5) / (ms5 * 1e-3) / 1e9
                    sweep.append({"n": n_, "kkt_ms": ms5, "kkt_gbs": gbs, "kkt_frac_of_hbm_peak": gbs / peak,
                                  "solves_per_s": int((o5["status"] == 0).sum()) / t5})
                    s5.close()
                extra["cfg5_horizon_sweep_b2048"] = sweep
            except Exception as e:
                extra["cfg3_cfg5_error"] = repr(e)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    value = conv_total * args.steps / el
    e2e_value = conv_e2e_total * m["e2e_steps"] / el_e2e
    line = {
        "metric": metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": el / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload, "config_id": cid, "batch_per_gpu": B, "global_batch": B * world, "horizon_n": N,
                   "parallelism": f"instances sharded over {world} GPU(s), NCCL all-gather of u* (step i) beside the solve of step i+1" if world > 1 else "1 GPU",
                   "l2": "flushed between steps (a batch's working set fits in the 126 MB L2)",
                   "converged_fraction": conv_total / float(B * world), "mean_ipm_iterations": m["iters_mean"],
                   "solve": "one persistent kernel per step: a CTA owns an instance from the initial guess to convergence; the CTAs "
                            "sharing an SM enter the phases of an iteration together (instruction-cache locality)",
                   "gate_wait_ms_per_cta": m["stats"]["gate_ms"] / max(1, args.steps),
                   "queue_order": "longest first by the iteration counts the same slots needed in the previous step (every step of the bench "
                                  "solves the same instances: an exact hint; the warm-up steps build it); configs.index_order = without"},
        "roofline": roofline,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(m["h2d"]), "d2h_bytes_per_step": int(m["d2h"])},
        "gpu_launches": int(st["launches_total"]),
        "kernel_ms": dict(zip(["init", "associate", "eval", "kkt", "linesearch"], [x / args.steps for x in st["ms"]])),
        "kernel_ms_note": "mean time a CTA of the persistent solve kernel spends in each phase per step (SM cycle counters of the kernel)",
        "timing": "CUDA events on the work stream around the K steps (max over ranks)",
        "clocks": m["clocks"],
        "configs": extra,
    }
    if not args.no_cpu_baseline and world == 1:
        v, n, conv, secs = cpu_arm(cfg, lambda n_: configs.generate(cid, n_, n=n_h), 20.0, threads)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "cores_detail": cores_info, "kind": "port",
                                "sample": f"{n} instances of the same workload ({conv} converged) in {secs:.1f} s, "
                                          "CPU oracle (same algorithm, plain C, one instance per thread)"}
    elif world > 1:
        line["cpu_baseline"] = None
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
