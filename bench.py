#!/usr/bin/env python3
"""bench.py -- converged IK solves/sec on the BASELINE.json headline workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dtype f64|f32] [--batch B]
                    [--dump-outputs DIR]

Workload (`config`, identical in both arms): Cassie feet+pelvis IK (pelvis Full + LeftFootFront / RightFootFront
Position, world frame), library-default solver parameters (max_iterations 100, damping 1e-2, step 1.0), batch 65,536
seeded random reachable targets PER GPU (weak scaling: rank r solves problem indices [r*B, (r+1)*B)), FP64.

A "step" = one batched ik::dls over one batch of B problems.
  value     K timed steps through the pipelined queue (ikb_queue_*, include/ikb200.h): `--merge` consecutive batches, each
            with its own buffers, share ONE BULK launch, and the stragglers a launch leaves suspended when its ticket
            queue runs dry (a problem that never converges runs all 100 steps, dls.cpp:14) are continued by the NEXT
            group's launch beside its fresh problems; the last group's stragglers get one TAIL launch, inside the timed
            region.  Inputs resident in HBM, CUDA events, max over ranks.  `details.isolated_ms_per_batch` = the same
            steps through the plain per-batch call, one BULK + TAIL kernel pair per batch.
  e2e       the same metric through the HOST entry point (ikb_queue_submit_host / ikb_queue_wait): every step's inputs are
            copied from pinned host memory and its results are copied back and read inside the timed region.  The wire
            format is what a caller of the reference supplies and receives (cassie.cpp:95-113): per problem the pelvis pose
            as quaternion + translation and two foot positions (compact targets, 13 scalars), ONE shared initial guess
            (the workload's q0 is the same standing pose for every problem, SURVEY 8d), q and the success flag back --
            289 B per solve.  `e2e.full_io` is the round-1 format (SE3 targets, a q0 per problem, iters and resid read
            back: 669 B per solve).
  roofline  compute roofline of the solve: algorithmic FLOPs (SURVEY.md 8d: F_iter per evaluation x (iterations + 1)
            evaluations per converged problem) / event-timed device time, against the FP64 (FP32) FMA-pipe peak measured
            in this run (MEASURED_PEAKS.json has no vector-pipe figure; nominal 37.2 / 74.4 TFLOP/s beside it).
  configs   the other BASELINE.json configs (FP32, 4,096, humanoid 262,144, manipulator 1,048,576, single-solve latency,
            the table-driven kernel), each a lone batch with its own roofline fraction -- outside the headline timing.
  strong    the SAME global batch (65,536 Cassie; 1,048,576 manipulator) cut over the N ranks (SURVEY 8e).
  cpu_baseline / --impl reference: the restated reference CPU path (oracle/, "port": Pinocchio / Eigen are unavailable so
            the reference itself cannot be built), all host cores; that arm imports nothing from the product.

--dump-outputs DIR writes what the headline path returned for its last timed step (rank 0's batch) as DIR/<name>.npy:
q (nq x B), success, iters and resid, all in the solve's float type.  The inputs are seeded, so two builds run with the
same arguments can be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# dram__bytes_read.sum + dram__bytes_write.sum per FP64 step, from the committed ncu --set full capture of this command
# (profiles/r2_s10_merged_full.txt): one merged BULK launch of 8 steps, stragglers of the previous one included, moves 320.0 + 107.5 MB -> 53.4 MB per step
NCU_TRAFFIC_BYTES_F64 = 53.4e6
METRIC = "converged IK solves/sec (Cassie, batch 65,536)"
UNIT = "solves/s"
NOMINAL_TFLOPS = {"f64": 37.2, "f32": 74.4}


def static_config(batch, world, dtype):
    """The workload description both arms print verbatim (the driver compares `config` between them)."""
    return {"workload": "Cassie feet+pelvis IK (pelvis Full + 2 foot Position tasks, world frame), seeded random reachable targets, "
                        "q0 = SRDF standing pose, library defaults max_it=100 damping=1e-2 step=1.0",
            "batch_per_gpu": batch, "global_batch": batch * world, "dtype": dtype, "seed": 12345}


def hbm_bytes_per_solve(nq, tsz, s):
    # (q0 + targets) in, (q + resid) + success(1) + iters(4) out -- SURVEY 8d "Layout"
    return (nq + tsz) * s + (nq + 1) * s + 1 + 4


DUMP_LIMIT_BYTES = 63 << 20   # array data of --dump-outputs: with the .npy headers, under 64 MB in all


def dump_outputs(out_dir, outputs, dtype):
    """Writes each output array (batch along the last axis) as <out_dir>/<name>.npy in `dtype`.  When they exceed
    DUMP_LIMIT_BYTES, a fixed, seeded sample of problems is written instead, with their batch indices in index.npy."""
    arrays = {k: np.asarray(v).astype(dtype) for k, v in outputs.items()}
    B = arrays["success"].shape[-1]
    per_problem = sum(a.nbytes for a in arrays.values()) // B
    if per_problem * B > DUMP_LIMIT_BYTES:
        n = DUMP_LIMIT_BYTES // (per_problem + 8)
        idx = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
        arrays = {k: a[..., idx] for k, a in arrays.items()}
        arrays["index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def f_iter(model, pb):
    """SURVEY.md 8d: algorithmic FLOPs of one evaluate + solve + step (mul, add = 1, FMA = 2; column supports only; Gram
    and solve dense in m x nv).  Cassie feet+pelvis: 9,360."""
    n_rev = sum(1 for t in model.jtypes[1:] if t != 1)
    n_ff = sum(1 for t in model.jtypes[1:] if t == 1)
    nv, nq = model.nv, model.nq
    m = sum(int(t.dimension()) for _, t, _ in pb._tasks)
    fk = 81 * n_rev + 30 * n_ff
    jac = logs = 0
    ident = np.concatenate([np.eye(3).reshape(-1), np.zeros(3)])
    for _, t, _ in pb._tasks:
        if not hasattr(t, "frame"):
            continue
        f = model.getFrameId(t.frame)
        if not np.array_equal(np.asarray(model.framePlacements[f]), ident):
            fk += 18
        j, k_rev, ff = int(model.frame_parents[f]), 0, 0
        while j > 0:
            if model.jtypes[j] == 1:
                ff = 1
            else:
                k_rev += 1
            j = int(model.parents[j])
        k_cols = k_rev + 6 * ff
        dim = int(t.dimension())
        jac += 42 * k_rev + 100 * ff
        logs += 305 + (48 if dim == 6 else 33) * k_cols
    solve = m * (m + 1) // 2 * (2 * nv - 1) + m + m ** 3 / 3.0 + 2 * m * m + 2 * m * nv + nv
    step = 155 * n_ff + 2 * nv + 2 * nq + 2 * m
    return float(fk + jac + logs + solve + step)


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU while the timed region runs (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = threading.Event()
        self.armed = threading.Event()   # samples are recorded only while the timed region runs
        self.ready = threading.Event()   # NVML initialised (takes longer than a whole timed region)
        self.sm = []
        self.reasons = set()
        self.max_mhz = None
        self.power = []

    def run(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
            }
            self.ready.set()
            while not self.stop_flag.is_set():
                if not self.armed.is_set():
                    time.sleep(0.0005)
                    continue
                self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
                except Exception:
                    pass
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.001)
        except Exception as e:  # pragma: no cover
            self.reasons.add("sampler_error:%s" % type(e).__name__)
            self.ready.set()

    def summary(self):
        sm = sorted(self.sm)
        return {"sm_mhz": (sm[len(sm) // 2] if sm else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(sm),
                "power_w_max": (max(self.power) if self.power else None)}


def cpu_reference_arm(B_sample, steps, warmup, cores):
    """Times the restated reference CPU path (oracle) on a bounded sample of the workload, all host cores.  Imports
    nothing from the product: the problem and its targets come from oracle/workload.py."""
    from oracle import oracle as O
    from oracle import workload as OW

    opb, q0, tg = OW.cassie_feet_pelvis(B_sample)
    for _ in range(warmup):
        O.dls_batch(opb, q0[:256], tg[:256], nthreads=cores)
    t0 = time.perf_counter()
    conv = 0
    for _ in range(steps):
        _, ok, it, _ = O.dls_batch(opb, q0, tg, nthreads=cores)
        conv += int(ok.sum())
    dt = time.perf_counter() - t0
    return conv / dt, dt / steps * 1e3, float(ok.mean()), float(it.mean())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=48)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"])
    ap.add_argument("--batch", type=int, default=65536, help="problems per GPU per step")
    ap.add_argument("--cpu-sample", type=int, default=0, help="problems in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the `configs` / `strong` / product multi-GPU sections")
    ap.add_argument("--merge", type=int, default=8, help="consecutive batches per kernel pair in the pipelined queue (1 = off)")
    ap.add_argument("--depth", type=int, default=24, help="batches in flight in the pipelined queue")
    ap.add_argument("--e2e-merge", type=int, default=4, help="the same for the host-buffer (e2e) arm: smaller groups keep the "
                    "PCIe pipeline's fill / drain short")
    ap.add_argument("--e2e-depth", type=int, default=12, help="three groups in flight: host batches carry their stragglers too (ikb_queue_create)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write q, success, iters and resid of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = os.cpu_count() or 1
    config = static_config(args.batch, world, args.dtype)

    if args.impl == "reference":
        if rank != 0:
            return 0
        sample = args.cpu_sample or args.batch
        warm = max(args.warmup, 1)
        val, ms, conv_frac, mean_it = cpu_reference_arm(sample, args.steps, warm, cores)
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                                 "sample": "%d problems x %d steps of the same seeded workload; restated reference CPU "
                                           "path (Pinocchio/Eigen unavailable here), pthreads over all cores"
                                           % (sample, args.steps)},
                "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "details": {"sample": "%d problems per step" % sample, "converged_fraction": conv_frac, "mean_iterations": mean_it}}
        print(json.dumps(line))
        return 0

    import torch

    import ik_b200 as ik
    from ik_b200 import _capi as capi
    from ik_b200 import workloads as W

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    if world > 1:
        import torch.distributed as dist

        # rank 0 prints ONE JSON line on stdout: NCCL's own log (version banner, rings -- what the driver's rank check
        # reads) goes to stderr instead of being silenced
        os.environ.setdefault("NCCL_DEBUG", "INFO")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    tdt = torch.float64 if args.dtype == "f64" else torch.float32
    npdt = np.float64 if args.dtype == "f64" else np.float32
    itemsize = np.dtype(npdt).itemsize
    B = args.batch

    def pinned_array(shape, dtype):
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        ptr = capi.lib.ikb_host_alloc(max(n, 1))
        if not ptr:
            raise MemoryError("ikb_host_alloc failed")
        return np.frombuffer((C.c_char * n).from_address(ptr), dtype=dtype).reshape(shape)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def build_sets(pb, nB, nsets, start, dt, seed0=12345, b0=0):
        """`nsets` distinct seeded batches of nB problems on the device (targets = GPU FK of sampled configurations)."""
        m = pb.model()
        names = W.task_frames(pb)
        out = []
        for s in range(nsets):
            qstar = W.sample_configurations(m, nB, seed=seed0 + s, b0=b0)
            poses_t = torch.cat([ik.fk_batch(pb, torch.tensor(qstar[i:i + 65536].T.copy(), device=dev), names)
                                 for i in range(0, nB, 65536)], dim=1)
            poses = {n: poses_t[12 * i:12 * i + 12].T.cpu().numpy() for i, n in enumerate(names)}
            tg = W.targets_from_frame_poses(pb, poses, qstar)
            q0 = (np.tile(W.standing_configuration(m, W.CASSIE_STANDING), (nB, 1)) if start == "standing" else W.near_start(m, qstar))
            o = {"q": torch.empty((m.nq, nB), dtype=dt, device=dev), "success": torch.empty(nB, dtype=torch.uint8, device=dev),
                 "iters": torch.empty(nB, dtype=torch.int32, device=dev), "resid": torch.empty(nB, dtype=dt, device=dev)}
            out.append((torch.tensor(q0.T.copy(), dtype=dt, device=dev), torch.tensor(tg.T.copy(), dtype=dt, device=dev), o, tg, q0))
        return out

    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def time_lone(pb, sets, prm, steps, warm=3, solve=None):
        """Lone batches through the per-batch call: CUDA-event time per batch, L2 flushed between timed launches."""
        solve = solve or (lambda p, q, t, o: ik.dls_batch(p, q, t, prm, o))
        for w in range(warm):
            s = sets[w % len(sets)]
            solve(pb, s[0], s[1], s[2])
        torch.cuda.synchronize()
        tot = 0.0
        for k in range(steps):
            s = sets[k % len(sets)]
            flush_buf.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            solve(pb, s[0], s[1], s[2])
            e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        o = sets[(steps - 1) % len(sets)][2]
        it = o["iters"].to(torch.int64)
        ok = o["success"].to(torch.int64)
        return tot / steps, int(ok.sum().item()), int((it + ok).sum().item()), float(it.double().mean().item())

    pb = W.cassie_feet_pelvis_problem()
    pb.finalize(local_rank)
    m = pb.model()
    nq, tsz = m.nq, pb.target_size
    F_ITER = f_iter(m, pb)
    q0_np = np.tile(W.standing_configuration(m, W.CASSIE_STANDING), (B, 1))

    # Distinct input/output sets, rotated every step, so the per-step inputs are not L2 hits left by the previous
    # step: NSETS * (inputs+outputs) > 126 MB of L2.
    per_set = B * hbm_bytes_per_solve(nq, tsz, itemsize)
    nsets = max(2, int(np.ceil(160e6 / per_set)) + 1, args.depth)  # ... and no set twice among the batches in flight
    sets = build_sets(pb, B, nsets, "standing", tdt, b0=rank * B)
    prm = ik.dls_parameters()

    # ---- device-resident arm ----
    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.ready.wait(10.0)
    for w in range(args.warmup):
        q0_d, tg_d, out = sets[w % nsets][:3]
        ik.dls_batch(pb, q0_d, tg_d, prm, out)
    barrier()
    iso = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    iso[0].record()
    for k in range(args.steps):
        q0_d, tg_d, out = sets[k % nsets][:3]
        ik.dls_batch(pb, q0_d, tg_d, prm, out)
    iso[1].record()
    barrier()
    isolated_ms = iso[0].elapsed_time(iso[1]) / args.steps

    depth = max(args.depth, args.merge)
    queue = ik.SolveQueue(pb, depth, args.merge, local_rank)
    for w in range(max(args.warmup, args.merge)):
        q0_d, tg_d, out = sets[w % nsets][:3]
        queue.submit(q0_d, tg_d, prm, out)
    queue.drain()
    barrier()
    sampler.armed.set()
    launches0 = ik.kernel_launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()                       # the queue's compute stream waits for this point of the current stream
    last = None
    for k in range(args.steps):
        q0_d, tg_d, out = sets[k % nsets][:3]
        last, _ = queue.submit(q0_d, tg_d, prm, out)
    queue.flush()
    for t in range(max(0, last - depth + 1), last + 1):
        queue.wait_on_stream(t)          # ... and the current stream waits for every batch still in flight
    ev[1].record()
    barrier()
    queue.drain()
    launches = ik.kernel_launch_count() - launches0
    elapsed_ms = ev[0].elapsed_time(ev[1])
    sampler.armed.clear()
    # the later sections reuse these output buffers
    last_outputs = None
    if args.dump_outputs and rank == 0:
        last_outputs = {k: v.cpu().numpy() for k, v in sets[(args.steps - 1) % nsets][2].items()}

    # optional final result gather (SURVEY 8e): not part of the solve, timed and reported separately
    gather_ms = None
    if world > 1:
        from ik_b200.sharding import gather_results

        last_out = sets[(args.steps - 1) % nsets][2]
        loc = {k: last_out[k] for k in ("q", "success", "iters")}
        gather_results(loc, B * world, dist)      # warm-up (NCCL communicator set-up)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        gather_results(loc, B * world, dist)
        g1.record()
        barrier()
        gather_ms = g0.elapsed_time(g1)
    it_last = sets[(args.steps - 1) % nsets][2]["iters"].float()
    it_hist = {"p50": it_last.quantile(0.5).item(), "p90": it_last.quantile(0.9).item(), "p95": it_last.quantile(0.95).item(),
               "p99": it_last.quantile(0.99).item(), "at_max_iterations": (it_last >= 100).float().mean().item()}
    conv = evals = it_sum = 0
    for k in range(args.steps):
        out = sets[k % nsets][2]
        conv += int(out["success"].sum().item())
        it = out["iters"].to(torch.int64)
        it_sum += int(it.sum().item())
        # evaluations: a converged problem evaluated (iters+1) times, a failed one `iters` times
        evals += int((it + out["success"].to(torch.int64)).sum().item())

    # ---- e2e arm: HOST buffers through the queue's host entry point; the copies of one group of batches run beside the
    # kernels of its neighbours.  Headline wire format: compact targets, one shared q0, q + success back. ----
    e2e_depth = max(args.e2e_depth, args.e2e_merge)
    queue_h = ik.SolveQueue(pb, e2e_depth, args.e2e_merge, local_rank)
    # the round-1 wire format (669 B per solve) is bound by the link, not by the kernels: two groups in flight keep the copy
    # pipeline's fill / drain short (and a queue this shallow launches a TAIL per host group instead of carrying)
    full_depth = max(8, args.e2e_merge)
    queue_f = ik.SolveQueue(pb, full_depth, args.e2e_merge, local_rank)
    nbuf = e2e_depth
    csz = pb.compact_target_size
    host_tg = [np.ascontiguousarray(sets[s][3], dtype=np.float64) for s in range(min(nsets, 3))]
    h_q0 = [pinned_array((nq, B), npdt) for _ in range(nbuf)]
    h_tg = [pinned_array((tsz, B), npdt) for _ in range(nbuf)]
    h_ctg = [pinned_array((csz, B), npdt) for _ in range(nbuf)]
    h_outs = [{"q": pinned_array((nq, B), npdt), "success": pinned_array((B,), np.uint8),
               "iters": pinned_array((B,), np.int32), "resid": pinned_array((B,), npdt)} for _ in range(nbuf)]
    for i in range(nbuf):
        h_q0[i][:] = q0_np.T
        h_tg[i][:] = host_tg[i % len(host_tg)].T
        h_ctg[i][:] = pb.compact_targets(host_tg[i % len(host_tg)]).T
    h_q0_one = pinned_array((nq,), npdt)
    h_q0_one[:] = q0_np[0]
    e2e_steps = args.steps
    lag = max(1, e2e_depth - 1)              # results of step k are consumed after step k + lag has been submitted

    def e2e_run(nsteps, lean):
        got = 0
        tickets = []
        qh = queue_h if lean else queue_f
        lg = lag if lean else max(1, full_depth - 1)
        for k in range(nsteps):
            i = k % nbuf
            if lean:
                t, _ = qh.submit_host(h_q0_one, h_ctg[i], prm, args.dtype, "soa", h_outs[i], compact=True, outputs=("q", "success"))
            else:
                t, _ = qh.submit_host(h_q0[i], h_tg[i], prm, args.dtype, "soa", h_outs[i])
            tickets.append(t)
            if k >= lg:
                qh.wait(tickets[k - lg])
                got += int(h_outs[(k - lg) % nbuf]["success"].sum())
        for k in range(max(0, nsteps - lg), nsteps):
            qh.wait(tickets[k])
            got += int(h_outs[k % nbuf]["success"].sum())
        return got

    e2e_run(nbuf + args.e2e_merge, False)    # every slot's staging buffers exist before the timed regions
    e2e_run(nbuf + args.e2e_merge, True)
    for k in range(2):
        ik.dls_batch_host(pb, h_q0[0], h_tg[0], prm, args.dtype, "soa", h_outs[0])
    t0 = time.perf_counter()
    for k in range(3):
        ik.dls_batch_host(pb, h_q0[0], h_tg[0], prm, args.dtype, "soa", h_outs[0])
    e2e_isolated_ms = (time.perf_counter() - t0) / 3 * 1e3
    barrier()
    sampler.armed.set()  # the clocks record covers both timed regions (device-resident steps and e2e steps)
    t0 = time.perf_counter()
    e2e_conv = e2e_run(e2e_steps, True)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    t0 = time.perf_counter()
    full_conv = e2e_run(e2e_steps, False)
    torch.cuda.synchronize()
    full_s = time.perf_counter() - t0
    sampler.armed.clear()
    sampler.stop_flag.set()
    sampler.join()
    barrier()

    # ---- the other BASELINE configs, strong scaling, the in-product multi-GPU handle (outside the headline timing) ----
    peak64, peak32 = C.c_double(0), C.c_double(0)
    capi.check(capi.lib.ikb_measure_fma_peak(capi.F64, local_rank, C.byref(peak64)), "ikb_measure_fma_peak")
    capi.check(capi.lib.ikb_measure_fma_peak(capi.F32, local_rank, C.byref(peak32)), "ikb_measure_fma_peak")
    peaks = {"f64": peak64.value, "f32": peak32.value}
    extras, strong, product_multi = {}, {}, None

    def entry(name, pbx, setsx, dt_name, steps, fi, note, solve=None, prmx=None):
        ms, cv, ev_, mean_it = time_lone(pbx, setsx, prmx or prm, steps, solve=solve)
        nB = setsx[0][0].shape[1]
        tf = fi * ev_ / (ms * 1e-3) / 1e12
        extras[name] = {"value": cv / (ms * 1e-3), "unit": UNIT, "batch": nB, "dtype": dt_name, "ms_per_batch": ms, "kernel": pbx.kernel_name(dt_name),
                        "converged_fraction": cv / nB, "mean_iterations": mean_it, "f_iter": fi,
                        "roofline": {"bound": "%s_fma_pipe" % ("fp64" if dt_name == "f64" else "fp32"), "achieved": tf,
                                     "peak": peaks[dt_name], "unit": "TFLOP/s", "frac": tf / peaks[dt_name]}, "note": note}
        return cv, ev_

    def queued_entry(name, pbx, setsx, dt_name, fi, cv, ev_, merge, nst):
        """The same batches through the pipelined queue (`merge` per BULK launch, stragglers carried): adds queued_* to
        extras[name].  One set per batch in flight -- a carried straggler lives in its batch's output buffers."""
        depth = 2 * merge
        assert len(setsx) >= depth
        qx = ik.SolveQueue(pbx, depth, merge, local_rank)
        for w in range(depth):
            sx = setsx[w % len(setsx)]
            qx.submit(sx[0], sx[1], prm, sx[2])
        qx.drain()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        lastt = None
        for k in range(nst):
            sx = setsx[k % len(setsx)]
            lastt, _ = qx.submit(sx[0], sx[1], prm, sx[2])
        qx.flush()
        for t in range(max(0, lastt - depth + 1), lastt + 1):
            qx.wait_on_stream(t)
        e1.record()
        torch.cuda.synchronize()
        qx.drain()
        qms = e0.elapsed_time(e1) / nst
        tf = fi * ev_ / (qms * 1e-3) / 1e12
        extras[name].update({"queued_ms_per_batch": qms, "queued_value": cv / (qms * 1e-3), "queued_roofline_frac": tf / peaks[dt_name],
                             "queued_note": "%d timed batches through ikb_queue, %d per BULK launch, stragglers carried into the next launch, "
                                            "final TAIL inside the timed region" % (nst, merge)})

    if not args.no_extras and rank == 0:
        lone = "one lone batch per launch (per-batch call, L2 flushed between launches)"
        if args.dtype == "f64":
            entry("cassie_65536_f64_lone", pb, sets[:4], "f64", 6, F_ITER, lone)
        sets32 = build_sets(pb, 65536, 3, "standing", torch.float32)
        entry("cassie_65536_f32", pb, sets32, "f32", 6, F_ITER, lone + "; FP32 instantiation (north_star 1e-4 rad: met by 99.4 % of the problems, "
              "as by the reference's own arithmetic in float -- tests/test_oracle_f32.py)")
        del sets32
        entry("cassie_4096_f64", pb, build_sets(pb, 4096, 8, "standing", torch.float64), "f64", 8, F_ITER, lone + "; BASELINE config 2 (latency configuration: team-per-problem kernel)")
        hpb = W.humanoid_problem()
        hpb.finalize(local_rank)
        hsets = build_sets(hpb, 262144, 4, "near", torch.float64)
        hcv, hev = entry("humanoid_262144_f64", hpb, hsets, "f64", 4, f_iter(hpb.model(), hpb),
                         lone + "; BASELINE config 4, warm-started (W.near_start)")
        queued_entry("humanoid_262144_f64", hpb, hsets, "f64", f_iter(hpb.model(), hpb), hcv, hev, 2, 8)
        del hsets
        mpb = W.manipulator_problem()
        mpb.finalize(local_rank)
        msets = build_sets(mpb, 1048576, 2, "near", torch.float64)
        entry("manipulator_1048576_f64", mpb, msets, "f64", 3, f_iter(mpb.model(), mpb), lone + "; BASELINE config 5 on ONE GPU, warm-started, 7-DoF")
        # the table-driven team-per-problem kernel (dls_coop.cuh): what ANY robot / task mix without a compiled specialisation gets
        os.environ["IKB_FORCE_GENERIC"] = "1"
        try:
            gpb = W.cassie_feet_pelvis_problem()
            gpb.finalize(local_rank)
            entry("table_driven_cassie_65536_f64", gpb, sets[:4], "f64", 4, F_ITER, lone + "; the same workload forced off its specialisation")
            ppb = W.cassie_demo_posture_problem()
            ppb.finalize(local_rank)
            psets = build_sets(ppb, 65536, 2, "standing", torch.float64)
            entry("table_driven_demo_posture_65536_f64", ppb, psets, "f64", 3, f_iter(ppb.model(), ppb), lone + "; the demo's full task set (26 rows, 2 levels), ik::dls")
            pprm = ik.pik_parameters(lambdas=[1e-2, 1e-1])
            entry("pik_demo_posture_65536_f64", ppb, psets, "f64", 2, f_iter(ppb.model(), ppb), lone + "; ik::pik on the same task set (roofline vs the DLS FLOP count)",
                  solve=lambda p, q, t, o: ik.pik_batch(p, q, t, pprm, o))
            del psets
        finally:
            os.environ.pop("IKB_FORCE_GENERIC", None)
        # single-solve latency through the reference's own call shape (ik::dls on one problem; BASELINE config 1's counterpart)
        q0_1 = W.standing_configuration(m, W.CASSIE_STANDING)
        tg_1 = sets[0][3][0]
        for name, t, _ in pb._tasks:
            off = pb.target_offset(t)
            t.target[:] = tg_1[off:off + 12]
        data = ik.dls_data(pb)
        for _ in range(5):
            ik.dls(pb, q0_1, data)
        t0 = time.perf_counter()
        nrep = 50
        for _ in range(nrep):
            ik.dls(pb, q0_1, data)
        lat_ms = (time.perf_counter() - t0) / nrep * 1e3
        it_default = data.iterations
        demo_prm = ik.dls_parameters(max_iterations=200, step_length=0.1, damping=0.1)
        t0 = time.perf_counter()
        for _ in range(20):
            ik.dls(pb, q0_1, data, p=demo_prm)
        lat_demo_ms = (time.perf_counter() - t0) / 20 * 1e3
        extras["single_solve_latency"] = {"ms": lat_ms, "iterations": it_default,
                                          "demo_params_ms": lat_demo_ms, "demo_params_iterations": data.iterations,
                                          "api": "ik.dls -> ikb_dls_solve_ex (host call: H2D, one team on the table-driven kernel, D2H of q/dq/e/J, sync)",
                                          "note": "the reference's demo ticks at 50 Hz = 20 ms (cassie.cpp:148)"}

    # strong scaling: the SAME global batch cut over the ranks (rank r solves [r B/G, (r+1) B/G)); every rank times its
    # slice, the job time is the max over ranks
    def strong_entry(name, pbx, Bglob, start):
        nloc = Bglob // world
        setsx = build_sets(pbx, nloc, 8, start, torch.float64, b0=rank * nloc)   # one per batch in flight (depth 8): a carried
        #                                                                         straggler lives in its batch's output buffers
        barrier()
        ms, cv, _, _ = time_lone(pbx, setsx, prm, 5)
        qx = ik.SolveQueue(pbx, 8, 4, local_rank)
        for w in range(8):
            s = setsx[w % len(setsx)]
            qx.submit(s[0], s[1], prm, s[2])
        qx.drain()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        lastt = None
        nst = 16
        for k in range(nst):
            s = setsx[k % len(setsx)]
            lastt, _ = qx.submit(s[0], s[1], prm, s[2])
        qx.flush()
        for t in range(max(0, lastt - 7), lastt + 1):
            qx.wait_on_stream(t)
        e1.record()
        barrier()
        qx.drain()
        qms = e0.elapsed_time(e1) / nst
        st = torch.tensor([ms, qms], dtype=torch.float64, device=dev)
        sm = torch.tensor([cv], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(st, op=dist.ReduceOp.MAX)
            dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms_max, qms_max = st.tolist()
        strong[name] = {"global_batch": Bglob, "per_gpu": nloc, "lone_ms": ms_max, "lone_value": sm.item() / (ms_max * 1e-3),
                        "queued_ms": qms_max, "queued_value": sm.item() / (qms_max * 1e-3), "unit": UNIT, "kernel": pbx.kernel_name("f64"),
                        "note": "strong scaling: one global batch over %d GPU(s); lone = per-batch call, queued = ikb_queue merge 4; "
                                "max over ranks" % world}

    if not args.no_extras:
        strong_entry("cassie_65536", pb, 65536, "standing")
        mpb2 = W.manipulator_problem()
        mpb2.finalize(local_rank)
        strong_entry("manipulator_1048576", mpb2, 1048576, "near")
        barrier()
        # several GPUs through the PRODUCT (ikb_multi_*): one host thread on rank 0 shards a host batch of world x B problems
        # over all visible GPUs.  The other ranks must leave their GPUs idle meanwhile -- an NCCL barrier would keep a
        # spinning kernel on each of them -- so they wait on a file flag, on the CPU.
        flag = os.path.join(tempfile.gettempdir(), "ikb_bench_multi_done_%d_%s" % (os.getuid(), os.environ.get("MASTER_PORT", "0")))
        if rank == 0 and os.path.exists(flag):
            os.remove(flag)
        barrier()
        if rank == 0 and torch.cuda.device_count() >= max(world, 1):
            G = max(world, 1)
            multi = ik.MultiGPU(pb, devices=list(range(G)), depth=12, merge=4)
            Bm = B * G
            mq0 = pinned_array((nq,), np.float64)
            mq0[:] = q0_np[0]
            NB = 12                                  # host buffers = queue depth: three groups in flight (host batches carry)
            mtg = [pinned_array((csz, Bm), np.float64) for _ in range(NB)]
            mout = [{"q": pinned_array((nq, Bm), np.float64), "success": pinned_array((Bm,), np.uint8)} for _ in range(NB)]
            for i in range(NB):
                mtg[i][:] = np.tile(pb.compact_targets(host_tg[i % len(host_tg)]).T, (1, G))
            def mrun(n):
                got, tk = 0, []
                for k in range(n):
                    t, _ = multi.submit_host(mq0, mtg[k % NB], prm, "f64", "soa", mout[k % NB], compact=True, outputs=("q", "success"))
                    tk.append(t)
                    if k >= NB - 1:
                        multi.wait(tk[k - (NB - 1)])
                        got += int(mout[(k - (NB - 1)) % NB]["success"].sum())
                for k in range(max(0, n - (NB - 1)), n):
                    multi.wait(tk[k])
                    got += int(mout[k % NB]["success"].sum())
                return got
            mrun(NB + 4)
            t0 = time.perf_counter()
            got = mrun(24)
            ms_ = (time.perf_counter() - t0)
            product_multi = {"value": got / ms_, "unit": UNIT, "devices": G, "global_batch_per_step": Bm, "steps": 24,
                             "api": "ikb_multi_submit_host / ikb_multi_wait from ONE host thread (compact targets, shared q0, q + success back)",
                             "note": "measured on rank 0 while the other ranks idle; no collective, results land in the caller's host arrays"}
            del multi
        if rank == 0:
            open(flag, "w").close()
        else:
            t_wait = time.time()
            while not os.path.exists(flag) and time.time() - t_wait < 300:
                time.sleep(0.01)
        barrier()
        if rank == 0:
            os.remove(flag)

    # ---- reduce over ranks ----
    stats = torch.tensor([elapsed_ms, e2e_s, full_s], dtype=torch.float64, device=dev)
    sums = torch.tensor([conv, e2e_conv, evals, it_sum, full_conv], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    elapsed_ms_max, e2e_s_max, full_s_max = stats.tolist()
    conv_all, e2e_conv_all, evals_all, it_all, full_conv_all = sums.tolist()

    if rank == 0:
        value = conv_all / (elapsed_ms_max * 1e-3)
        e2e_value = e2e_conv_all / e2e_s_max
        k_ms = elapsed_ms / args.steps
        flops_per_launch = F_ITER * (evals / args.steps)
        achieved_tf = flops_per_launch / (k_ms * 1e-3) / 1e12
        peak = peaks[args.dtype]
        hbm_peak = None
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                hbm_peak = json.load(f).get("hbm_gbs")
        except Exception:
            pass
        hbm_src = "MEASURED_PEAKS.json" if hbm_peak else "fallback (B200_PROFILING.md)"
        hbm_peak = hbm_peak or 6650.0
        hbm_achieved = B * hbm_bytes_per_solve(nq, tsz, itemsize) / (k_ms * 1e-3) / 1e9
        cpu = None
        if not args.no_cpu_baseline:
            sample = args.cpu_sample or args.batch
            probe, _, _, _ = cpu_reference_arm(min(sample, 4096), 1, 1, cores)
            passes = int(min(50, max(1, np.ceil(10.0 * probe / sample))))
            v, ms, cf, mi = cpu_reference_arm(sample, passes, 1, cores)
            v1, _, _, _ = cpu_reference_arm(min(sample, 4096), 1, 0, 1)   # one thread, small sample (SURVEY 8d: both)
            cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "single_thread_value": v1,
                   "sample": "%d problems x %d passes of the same seeded workload (%.1f s); restated reference CPU path "
                             "(Pinocchio/Eigen unavailable), pthreads over all %d host cores"
                             % (sample, passes, passes * ms / 1e3, cores)}
        iso_evals = evals / args.steps
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": elapsed_ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": config,
            "details": {"kernel": pb.kernel_name(args.dtype),
                        "l2": "inputs/outputs rotate over %d distinct batches (%.0f MB > 126 MB L2)" % (nsets, nsets * per_set / 1e6),
                        "pipeline": "ikb_queue, depth %d, %d consecutive batches per BULK launch; stragglers carried into the next launch, "
                                    "one TAIL launch at the end" % (depth, args.merge),
                        "isolated_ms_per_batch": isolated_ms,
                        "isolated_value": conv / args.steps / (isolated_ms * 1e-3) * world,
                        "isolated_roofline_frac": F_ITER * iso_evals / (isolated_ms * 1e-3) / 1e12 / peak,
                        "converged_fraction": conv_all / (B * world * args.steps),
                        "mean_iterations": it_all / (B * world * args.steps), "iterations": it_hist,
                        "result_gather_ms": gather_ms, "f_iter": F_ITER},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int((B * csz + nq) * itemsize),
                    "d2h_bytes_per_step": int(B * (nq * itemsize + 1)), "steps": e2e_steps,
                    "bytes_per_solve": (csz * itemsize) + nq * itemsize + 1,
                    "api": "ikb_queue_submit_host + ikb_queue_wait (pinned host buffers; H2D, SE3 expansion, solve, D2H of every step)",
                    "wire_format": "compact targets (pelvis quaternion + translation, two foot positions: %d scalars), one shared q0, "
                                   "q + success read back -- what a caller of the reference supplies and receives" % csz,
                    "pipeline": "ikb_queue, depth %d, %d consecutive host batches per BULK launch; their stragglers are carried into the next "
                                "group's launch (depth >= 3 x merge), the copy-out of a group follows that launch; the SE3 expansion of the "
                                "compact targets runs on the compute stream" % (e2e_depth, args.e2e_merge),
                    "isolated_ms_per_batch": e2e_isolated_ms,
                    "isolated_api": "ikb_dls_solve_batch_host (blocking, one batch at a time, full_io format)",
                    "full_io": {"value": full_conv_all / full_s_max, "h2d_bytes_per_step": int(B * (nq + tsz) * itemsize),
                                "d2h_bytes_per_step": int(B * ((nq + 1) * itemsize + 5)), "bytes_per_solve": (2 * nq + tsz + 1) * itemsize + 5,
                                "note": "round-1 wire format: 12-scalar SE3 target per task, a q0 per problem, q + success + iters + resid back"}},
            "gpu_launches": int(launches),
            "roofline": {"bound": "fp64_fma_pipe" if args.dtype == "f64" else "fp32_fma_pipe",
                         "achieved": achieved_tf, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved_tf / peak if peak else None,
                         "traffic": NCU_TRAFFIC_BYTES_F64 if (args.dtype == "f64" and B == 65536) else None,
                         "traffic_source": "ncu --set full of this command, profiles/r2_s10_merged_full.txt: DRAM bytes of one merged BULK launch (8 steps + the stragglers carried over from the previous launch): (320.0 + 107.5 MB) / 8; algorithmic 43.8 MB",
                         "kernels": "one BULK launch of %s per group of %d steps, which also continues the stragglers the previous group left "
                                    "suspended; ONE TAIL launch when the queue runs empty; kernel_ms = device time of the timed region / steps"
                                    % (pb.kernel_name(args.dtype), args.merge),
                         "peak_source": "measured in this run (ikb_measure_fma_peak); nominal %.1f"
                                        % NOMINAL_TFLOPS[args.dtype],
                         "frac_of_nominal": achieved_tf / NOMINAL_TFLOPS[args.dtype],
                         "executed_pipe_busy_ncu": 0.40 if (args.dtype == "f64" and B == 65536) else None,
                         "executed_note": "`frac` counts ALGORITHMIC FLOPs (SURVEY 8d: the dense J J^T + LDL^T of the reference's step); the arrow "
                                          "step reaches the same dq with fewer executed FLOPs, so ncu's FP64-pipe utilisation of the merged launch "
                                          "(sm__pipe_fp64_cycles_active 39.5-39.9 %, profiles/r2_s15_merged_full.txt) is lower than `frac`",

                         "flops_per_launch": flops_per_launch, "kernel_ms": k_ms,
                         "hbm": {"achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": hbm_achieved / hbm_peak, "peak_source": hbm_src}},
            "cpu_baseline": cpu,
            "configs": extras or None,
            "strong": strong or None,
            "product_multi_gpu": product_multi,
            "clocks": sampler.summary(),
        }
        if last_outputs is not None:
            dump_outputs(args.dump_outputs, last_outputs, npdt)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
