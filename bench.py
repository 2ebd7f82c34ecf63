#!/usr/bin/env python
"""bench.py -- headline measurement of the hot path (see DESIGN.md "Measurement").

A *step* is one Levenberg-Marquardt iteration of the sliding-window BA (fused evaluate + J^T J
assembly, Schur elimination, reduced Cholesky, back-substitution, candidate cost, LM decision) on the
synthetic KITTI-shaped window of BASELINE.json configs[1] (stereo+IMU, 10 keyframes, 4000 landmarks per
GPU).  `value` = Jacobian-carrying residual rows processed per second with the problem resident in HBM;
`e2e` = the same through the public host API (problem upload from host buffers, K iterations, result
download).  Extra objects on the same JSON line:

  window20       north_star's target shape (20 keyframes, 8000 landmarks, 19 IMU factors), device-resident and e2e, with its own
                 CPU number (N = 1 only)
  roofline       the TwoFrame Jacobian-eval kernel at configs[4] scale: algorithmic bytes / CUDA-event time / measured HBM peak
  roofline_fused the kernel Solve actually launches for the visual factors (ba_linearize_kernel<0>), same scale, 52 B per block
  kernels        CUDA-event time of every kernel of one LM pass (window and map scale) -- compute vs all-reduce at N > 1
  global_ba      configs[4]-scale map BA (5000 keyframes, 500k landmarks), sharded by landmark, multifrontal reduced solve
  icp            configs[2]: 120k-point scan vs 1M-point map: points/s resident, e2e, kNN-only, roofline of the association kernel
  cpu_baseline   the oracle restatement of the Ceres / PCL path timed on the host cores (a reported baseline, not a target)

    python bench.py --gpus N --steps K --warmup W            # torchrun for N > 1
    python bench.py --impl reference ...                       # CPU oracle arm (rank 0 only)
    python bench.py --quick                                    # headline legs only (A/B runs)
    python bench.py --dump-outputs DIR                         # also write the headline window's solved parameters as .npy
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from lvio_fusion_b200 import backend, synth  # noqa: E402

N_KF, N_LM = 10, 4000                # configs[1]
W20_KF, W20_LM = 20, 8000            # configs[3]'s BA part = north_star's 20-keyframe target
ICP_K, ICP_P = 120000, 1000000       # configs[2]
EVAL_KF, EVAL_LM = 5000, 500000      # configs[4] scale
# dram__bytes_read.sum + dram__bytes_write.sum of one ba_eval_two_frame_kernel launch at that scale, from the `ncu --set full`
# capture summarised in profiles/eval_r1_v3_summary.txt (75.19 MB + 293.14 MB): a constant from that capture, not measured in-run
EVAL_DRAM_BYTES_PER_LAUNCH = 368.33e6
# the same for ba_linearize_kernel<0> at that scale: profiles/global_r2_final_summary.txt (143.74 MB read + 115.21 MB written)
FUSED_DRAM_BYTES_PER_LAUNCH = 258.95e6
BYTES_TWO_FRAME = 308                # SURVEY 8(d): 40 const + 12 idx + 16 r + 240 J
BYTES_FUSED = {0: 52, 1: 52, 2: 44}  # SURVEY 8(d) fused mode: TwoFrame, PoseOnly, TwoCamera
BYTES_KNN_QUERY = 40                 # query 16 + idx 12 + d2 12, plus 16 B per map point amortised over the queries
PER = 10                             # LM iterations per solve


def cpu_threads():
    n = os.cpu_count() or 1
    return min(8, max(1, int(0.75 * n)))       # the reference's own rule, estimator.cpp:10


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)["hbm_gbs"], "MEASURED_PEAKS.json"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    def __init__(self, device):
        super().__init__(daemon=True)
        self.device, self.rows, self.stop_flag = device, [], False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def bench_options(api, iters, threads=1):
    # fixed iteration count: tolerances off so both arms do exactly the same number of LM iterations
    return backend.default_options(api, max_num_iterations=iters, function_tolerance=0.0, gradient_tolerance=0.0,
                                   parameter_tolerance=0.0, num_threads=threads)


def run_solves(problem, d, api, total_iters, per_solve, threads=1):
    """Run LM iterations in solves of `per_solve` iterations restarted from the initial guess until
    `total_iters` iterations have been executed; returns iterations actually executed."""
    done = 0
    while done < total_iters:
        k = min(per_solve, total_iters - done)
        problem.update_params(d["poses"], d["vec3"], d["rho"])
        s = problem.solve(bench_options(api, k, threads))
        done += max(1, s.num_iterations)
    return done


def cpu_window(orc, octx, n_kf, n_lm, iters, T):
    d = synth.make_ba_problem(n_kf, n_lm, with_imu=True, seed=synth.SEED)
    p = backend.Problem.from_dict(octx, d)
    run_solves(p, d, orc, PER, PER, T)
    t0 = time.perf_counter()
    it = run_solves(p, d, orc, iters, PER, T)
    dt = time.perf_counter() - t0
    return synth.count_rows(d) * it / dt, it, dt


def cpu_icp(orc, octx, T):
    """All ICP_K queries against the full map: kd-tree build (the reference rebuilds it per call, association.cpp:278-279) + 3-NN +
    gate + 4 LM iterations."""
    sc = synth.make_icp_problem(ICP_K, ICP_P, seed=synth.SEED, kind="surf")
    fo = backend.FeatureAssociation(octx)
    orc.icp_set_threads(fo.h, T)
    e0 = synth.relative_rpyxyz(sc["map_pose"], sc["frame_pose"])
    t0 = time.perf_counter()
    fo.set_map(sc["map"], sc["cell_size"])
    t1 = time.perf_counter()
    fo.scan_to_map(sc["mode"], sc["scan"], sc["frame_pose"], sc["map_pose"], e0, sc["weight"], -1.0, sc["huber_a"], sc["thr"])
    t2 = time.perf_counter()
    return {"metric": "icp_points_per_s", "value": ICP_K / (t2 - t0), "unit": "points/s", "cores": T, "kind": "port",
            "tree_build_s": t1 - t0, "scan_to_map_s": t2 - t1,
            "sample": "all %d queries vs the %d-point map: kd-tree build + exact 3-NN + gate + 4 LM iterations, %d threads" % (ICP_K, ICP_P, T)}


def workload_text(rows):
    return ("configs[1]: KITTI-shaped stereo+IMU 10-keyframe window, %d landmarks per GPU (sharded by landmark, one in-kernel all-reduce of the "
            "reduced system over NVLink peer memory per iteration), %d residual rows total; step = one LM iteration" % (N_LM, rows))


def reference_arm(args):
    """CPU arm: the oracle restatement of the reference's Ceres+PCL path on the host cores."""
    from oracle import binding
    orc = binding.load()
    T = cpu_threads()
    octx = backend.Context(orc)
    d = synth.make_ba_problem(N_KF, N_LM * max(1, args.gpus), with_imu=True, seed=synth.SEED)     # the same (weak-scaled) window the GPU arm shards
    rows = synth.count_rows(d)
    p = backend.Problem.from_dict(octx, d)
    run_solves(p, d, orc, max(1, args.warmup), PER, T)
    t0 = time.perf_counter()
    it = run_solves(p, d, orc, args.steps, PER, T)
    dt = time.perf_counter() - t0
    val = rows * it / dt
    w20, it20, _ = cpu_window(orc, octx, W20_KF, W20_LM, 20, T)
    line = {
        "impl": "reference", "metric": "ba_residual_jacobian_rows_per_s", "value": val, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": it, "warmup": args.warmup, "ms_per_step": 1e3 * dt / it, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_text(rows), "blocks": synth.count_blocks(d), "iters_per_solve": PER},
        "cpu_baseline": {"value": val, "unit": "rows/s", "cores": T, "kind": "port",
                         "sample": "%d LM iterations of the full configs[1] window (oracle restatement of Ceres SPARSE_SCHUR, %d threads); the reference itself cannot be built here" % (it, T)},
        "window20": {"value": w20, "unit": "rows/s", "cores": T, "sample": "%d LM iterations of the 20-keyframe / %d-landmark window" % (it20, W20_LM)},
        "icp": cpu_icp(orc, octx, T),
        "e2e": {"value": val, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def kernel_split(lvb, run, iters):
    """CUDA-event time of every kernel of `run()` (direct launches, an event after each kernel on the launching stream):
    {kernel: microseconds per LM iteration}."""
    lvb.check(lvb.debug_timing(1), "debug_timing")
    run()
    buf = ctypes.create_string_buffer(1 << 20)
    lvb.check(lvb.debug_timing_report(buf, len(buf)), "debug_timing_report")
    acc = {}
    for ln in buf.value.decode().splitlines():
        name, us = ln.rsplit(" ", 1)
        name = name.strip("()")
        if name == "begin":
            continue
        acc[name] = acc.get(name, 0.0) + float(us)
    return {k: v / iters for k, v in acc.items()}


def dump_outputs(out_dir, problem):
    """What Problem.solve hands back to its caller: the solved parameter blocks (about 33 kB at configs[1])."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("poses", problem.poses()), ("vec3", problem.vec3()), ("inv_depths", problem.inv_depths())):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--quick", action="store_true", help="headline legs only")
    ap.add_argument("--skip-icp", action="store_true")
    ap.add_argument("--skip-roofline", action="store_true")
    ap.add_argument("--skip-global", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--blocks", type=int, default=0, help="repetitions of the timed region (0: enough for >= 50 solves); profiler runs use 1")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of the headline window returns to a caller "
                    "(poses, vec3, inverse depths of rank 0's shard) as DIR/<name>.npy in float64, to compare builds output for output")
    args = ap.parse_args()
    if args.quick:
        args.skip_icp = args.skip_roofline = args.skip_global = args.skip_cpu = True
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    from lvio_fusion_b200 import _capi
    lvb = _capi.load()
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        ctx = backend.Context(lvb, device=local_rank, stream=stream.cuda_stream)
        if world > 1:
            uid = ctypes.create_string_buffer(128)
            if rank == 0:
                lvb.check(lvb.comm_unique_id(uid), "comm_unique_id")
            box = [uid.raw]
            dist.broadcast_object_list(box, src=0)
            ctx.comm_init(rank, world, box[0])
        # rank-0-only legs run on their own world-1 context: on the communicator-attached one Problem.from_dict is a collective
        # (lvb_ba_finalize agrees on the unknown order and the envelope over the ranks) and would pair with nothing
        ctx1 = backend.Context(lvb, device=local_rank, stream=stream.cuda_stream) if world > 1 else ctx
        peak, peak_src = peaks()

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        def max_over_ranks(ms):
            if world == 1:
                return ms
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())

        def timed_blocks(fn, blocks):
            """`blocks` repetitions of fn(), each bracketed by barrier + synchronize and timed with CUDA events on the launching
            stream; returns the per-block times (max over ranks) and fn's last return value."""
            out, ret = [], None
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for _ in range(blocks):
                barrier()
                e0.record(stream)
                ret = fn()
                e1.record(stream)
                barrier()
                out.append(max_over_ranks(e0.elapsed_time(e1)))
            return out, ret

        def window_leg(c, n_kf, n_lm_per_gpu, steps, warmup):
            """Device-resident value + e2e of one window shape on context c (sharded by landmark when c is the communicator's)."""
            w = world if c is ctx else 1
            full = synth.make_ba_problem(n_kf, n_lm_per_gpu * w, with_imu=True, seed=synth.SEED)
            rows = synth.count_rows(full)
            d = synth.shard_ba_problem(full, rank, w) if w > 1 else full
            prob = backend.Problem.from_dict(c, d)
            run_solves(prob, d, lvb, max(3, warmup), PER)
            l0 = c.launch_count()
            its = run_solves(prob, d, lvb, steps, PER)
            launches = c.launch_count() - l0
            # the K-step timed region, repeated so that >= 50 solves stand behind the number; the median block is reported
            blocks = args.blocks if args.blocks > 0 else max(5, -(-50 * PER // max(1, steps)))
            times, its = timed_blocks(lambda: run_solves(prob, d, lvb, steps, PER), blocks)
            ms = float(np.median(times))
            res = {"rows": rows, "iters": its, "ms": ms, "launches": int(launches), "blocks": blocks,
                   "ms_min": float(np.min(times)), "ms_max": float(np.max(times)), "problem": prob, "data": d, "full": full}
            # e2e: build + upload + solve + download through the public API, host buffers
            h2d = sum(f[0].nbytes + f[1].nbytes for f in d["factors"].values()) + d["poses"].nbytes + d["vec3"].nbytes + d["rho"].nbytes + 22 * 8
            d2h = d["poses"].nbytes + d["vec3"].nbytes + d["rho"].nbytes

            def one_e2e():
                n = 0
                while n < steps:
                    p2 = backend.Problem.from_dict(c, d)
                    s2 = p2.solve(bench_options(lvb, PER))
                    p2.poses(); p2.vec3(); p2.inv_depths()
                    n += max(1, s2.num_iterations)
                    p2.close()
                return n
            one_e2e()
            walls = []
            for _ in range(max(3, blocks // 4)):
                barrier()
                t0 = time.perf_counter()
                n_it = one_e2e()
                barrier()
                walls.append(max_over_ranks((time.perf_counter() - t0) * 1e3))
            res.update({"e2e_ms": float(np.median(walls)), "e2e_iters": n_it, "h2d": int(h2d / PER), "d2h": int(d2h / PER)})
            return res

        # ---------------- BA headline: configs[1], weak scaling, N_LM landmarks per GPU, sharded by landmark (SURVEY 8e)
        sampler = ClockSampler(local_rank)
        sampler.start()
        w10 = window_leg(ctx, N_KF, N_LM, args.steps, args.warmup)
        sampler.stop_flag = True
        if args.dump_outputs and rank == 0:
            # the problem still holds the state its last timed solve left (the e2e part of the leg solves fresh problems)
            dump_outputs(args.dump_outputs, w10["problem"])
        value = w10["rows"] * w10["iters"] / (w10["ms"] * 1e-3)
        line = {
            "metric": "ba_residual_jacobian_rows_per_s", "value": value, "unit": "rows/s", "n_gpus": world, "steps": w10["iters"], "warmup": args.warmup,
            "ms_per_step": w10["ms"] / w10["iters"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_text(w10["rows"]),
                       "blocks": synth.count_blocks(w10["full"]), "iters_per_solve": PER,
                       "timing": "median of %d repetitions of the %d-step timed region (min %.4f / max %.4f ms per step)" % (w10["blocks"], w10["iters"], w10["ms_min"] / w10["iters"], w10["ms_max"] / w10["iters"]),
                       "l2": "BA working set (~3 MB) is L2-resident by design; the roofline legs stream 394 MB / 97 MB per launch (> 126 MB L2 together with their outputs)"},
            "e2e": {"value": w10["rows"] * w10["e2e_iters"] / (w10["e2e_ms"] * 1e-3), "unit": "rows/s", "h2d_bytes_per_step": w10["h2d"], "d2h_bytes_per_step": w10["d2h"],
                    "note": "Problem.from_dict (AoS->SoA, H2D) + solve(%d iterations) + D2H of all parameter blocks, per solve; bytes amortised per iteration" % PER},
            "gpu_launches": w10["launches"],
        }
        # per-kernel split of one pass (direct launches, CUDA event after every kernel): names the limiter at every N
        p10, d10 = w10["problem"], w10["data"]
        split = kernel_split(lvb, lambda: run_solves(p10, d10, lvb, PER, PER), PER)
        comm = sum(v for k, v in split.items() if "allreduce" in k.lower())
        line["kernels"] = {"window10_us_per_iteration": {k: round(v, 2) for k, v in sorted(split.items(), key=lambda kv: -kv[1])},
                           "compute_us": round(sum(split.values()) - comm, 2), "allreduce_us": round(comm, 2),
                           "note": "direct launches with an event after each kernel (the timed legs replay a CUDA graph); includes launch gaps"}
        # the only dense contraction of the path on the tensor cores (north_star: tcgen05 for the Schur reduce): same window, schur_mode = 1
        if world == 1:
            def run_tc(iters):
                n = 0
                while n < iters:
                    p10.update_params(d10["poses"], d10["vec3"], d10["rho"])
                    o = bench_options(lvb, PER); o.schur_mode = 1
                    n += max(1, p10.solve(o).num_iterations)
                return n
            run_tc(3 * PER)
            t_tc, it_tc = timed_blocks(lambda: run_tc(args.steps), 5)
            s_fp = p10.solve(bench_options(lvb, PER)); p10.update_params(d10["poses"], d10["vec3"], d10["rho"])
            o = bench_options(lvb, PER); o.schur_mode = 1
            s_tc = p10.solve(o)
            tc_split = kernel_split(lvb, lambda: run_tc(PER), PER)
            line["schur_tc"] = {"ms_per_step": float(np.median(t_tc)) / it_tc, "fp64_ms_per_step": w10["ms"] / w10["iters"],
                                "final_cost_rel_diff": abs(s_tc.final_cost - s_fp.final_cost) / s_fp.final_cost,
                                "us_per_iteration": {k: round(v, 2) for k, v in tc_split.items() if "schur" in k},
                                "note": "ba_schur_tc_kernel: tcgen05.mma kind::f16 on split-bf16 operands (hi/mid/lo), FP32 accumulation in TMEM, FP64 epilogue; "
                                        "opt-in (schur_mode = 1): the contraction is ~0.2 GFLOP per iteration, so packing + the FP64 scatter cost what the tensor pipe saves"}
        p10.close()

        # ---------------- north_star's target shape: 20 keyframes, 8000 landmarks, 19 IMU factors (N = 1)
        if world == 1 and not args.quick:
            w20 = window_leg(ctx1, W20_KF, W20_LM, args.steps, args.warmup)
            line["window20"] = {"metric": "ba_residual_jacobian_rows_per_s", "value": w20["rows"] * w20["iters"] / (w20["ms"] * 1e-3), "unit": "rows/s",
                                "ms_per_step": w20["ms"] / w20["iters"], "rows": w20["rows"],
                                "e2e": {"value": w20["rows"] * w20["e2e_iters"] / (w20["e2e_ms"] * 1e-3), "unit": "rows/s",
                                        "h2d_bytes_per_step": w20["h2d"], "d2h_bytes_per_step": w20["d2h"]},
                                "workload": "configs[3]'s BA part: stereo+IMU 20-keyframe window, %d landmarks, %d IMU factors" % (W20_LM, W20_KF - 1)}
            p20, d20 = w20["problem"], w20["data"]
            split20 = kernel_split(lvb, lambda: run_solves(p20, d20, lvb, PER, PER), PER)
            line["kernels"]["window20_us_per_iteration"] = {k: round(v, 2) for k, v in sorted(split20.items(), key=lambda kv: -kv[1])}
            p20.close()

        # ---------------- roofline of the dominant streaming kernel: TwoFrame Jacobian eval at configs[4] scale
        if rank == 0 and not args.skip_roofline:
            big = synth.make_ba_problem(EVAL_KF, EVAL_LM, with_imu=False, seed=synth.SEED)
            big["factors"] = {0: big["factors"][0]}
            pb = backend.Problem.from_dict(ctx1, big)
            nb = len(big["factors"][0][0])
            for _ in range(3):
                pb.evaluate_device(0)
            torch.cuda.synchronize()
            reps = 10
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
            ev[0].record(stream)
            for i in range(reps):
                pb.evaluate_device(0)
                ev[i + 1].record(stream)
            torch.cuda.synchronize()
            t_avg = sum(ev[i].elapsed_time(ev[i + 1]) for i in range(reps)) / reps
            ach = nb * BYTES_TWO_FRAME / (t_avg * 1e-3) / 1e9
            line["roofline"] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": EVAL_DRAM_BYTES_PER_LAUNCH,
                                "traffic_source": "profiles/eval_r1_v3_summary.txt (ncu --set full), not measured in-run",
                                "kernel": "ba_eval_two_frame_kernel", "blocks": nb, "bytes_per_block": BYTES_TWO_FRAME,
                                "us_per_launch": t_avg * 1e3, "peak_source": peak_src, "workload": "configs[4]-scale: %d keyframes, %d landmarks" % (EVAL_KF, EVAL_LM),
                                "rows_per_s": 2.0 * nb / (t_avg * 1e-3)}
            pb.close()

        # ---------------- configs[4]: map-scale global BA (banded reduced system), landmarks sharded over the ranks
        if not args.skip_global:
            g_full = synth.make_ba_problem(EVAL_KF, EVAL_LM, with_imu=True, seed=synth.SEED + 1)
            g_rows = synth.count_rows(g_full)
            g_blocks = synth.count_blocks(g_full)
            gd = synth.shard_ba_problem(g_full, rank, world) if world > 1 else g_full
            del g_full
            gp = backend.Problem.from_dict(ctx, gd)
            gp.solve(bench_options(lvb, 3))

            def g_solve():
                gp.update_params(gd["poses"], gd["vec3"], gd["rho"])
                return gp.solve(bench_options(lvb, 5))
            times, gs = timed_blocks(g_solve, 3)
            g_ms = float(np.median(times)) / max(1, gs.num_iterations)
            line["global_ba"] = {"metric": "ba_residual_jacobian_rows_per_s", "value": g_rows / (g_ms * 1e-3), "unit": "rows/s", "ms_per_iteration": g_ms,
                                 "iterations": gs.num_iterations, "rows": g_rows, "camera_dims": gp.dims()[0], "scaling": "strong",
                                 "cost": [gs.initial_cost, gs.final_cost],
                                 "workload": "configs[4]-scale: %d keyframes + IMU, %d landmarks, sharded by landmark; banded reduced camera system, multifrontal separator-tree Cholesky" % (EVAL_KF, EVAL_LM)}
            gsplit = kernel_split(lvb, g_solve, max(1, gs.num_iterations))
            line["kernels"]["global_ba_us_per_iteration"] = {k: round(v, 1) for k, v in sorted(gsplit.items(), key=lambda kv: -kv[1])}
            if world == 1:
                # the visual linearisation Solve launches: one launch covers the TwoFrame, PoseOnly and TwoCamera blocks (fused mode:
                # residuals and Jacobians never leave the chip); it runs once per accepted iteration
                us = gsplit.get("ba_linearize_kernel<0>")
                nblk = [len(gd["factors"][k][0]) for k in (0, 1, 2)]
                alg = sum(n * BYTES_FUSED[k] for k, n in zip((0, 1, 2), nblk))
                if us:
                    line["roofline_fused"] = {"bound": "hbm", "achieved": alg / (us * 1e-6) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / (us * 1e-6) / 1e9 / peak,
                                              "traffic": FUSED_DRAM_BYTES_PER_LAUNCH, "traffic_source": "profiles/global_r2_final_summary.txt (ncu --set full), not measured in-run",
                                              "kernel": "ba_linearize_kernel<0>", "blocks": nblk, "bytes_per_block": [BYTES_FUSED[k] for k in (0, 1, 2)],
                                              "us_per_launch": us, "peak_source": peak_src, "total_blocks": g_blocks,
                                              "note": "algorithmic bytes are SURVEY 8(d)'s fused-mode figures; the kernel also writes the per-factor coupling rows the Schur step reads"}
            gp.close()
            del gd

        # ---------------- ICP (configs[2]): points/s through scan_to_map, map resident vs e2e with set_map
        if not args.skip_icp:
            sc = synth.make_icp_problem(ICP_K, ICP_P, seed=synth.SEED, kind="surf")
            lo, hi = rank * ICP_K // world, (rank + 1) * ICP_K // world     # query tiles sharded, map replicated
            scan = sc["scan"][lo:hi]
            fa = backend.FeatureAssociation(ctx)
            e_init = synth.relative_rpyxyz(sc["map_pose"], sc["frame_pose"])
            fa.set_map(sc["map"], sc["cell_size"])
            argsicp = (sc["mode"], scan, sc["frame_pose"], sc["map_pose"], e_init, sc["weight"], -1.0, sc["huber_a"], sc["thr"])
            for _ in range(3):
                fa.scan_to_map(*argsicp)
            reps = 10
            times, _ = timed_blocks(lambda: [fa.scan_to_map(*argsicp) for _ in range(reps)], 3)
            icp_ms = float(np.median(times)) / reps
            walls = []
            for _ in range(3):
                barrier()
                t0 = time.perf_counter()
                fa.set_map(sc["map"], sc["cell_size"])
                fa.scan_to_map(*argsicp)
                barrier()
                walls.append(max_over_ranks((time.perf_counter() - t0) * 1e3))
            icp_e2e_ms = float(np.median(walls))
            line["icp"] = {"metric": "icp_points_per_s", "value": ICP_K / (icp_ms * 1e-3), "unit": "points/s", "ms_per_scan": icp_ms,
                           "e2e": {"value": ICP_K / (icp_e2e_ms * 1e-3), "unit": "points/s", "ms_per_scan": icp_e2e_ms,
                                   "note": "map upload + voxel build + scan upload + association + 4 LM iterations"},
                           "workload": "configs[2]: %d-point scan vs %d-point map, surf gate, Huber 0.1" % (ICP_K, ICP_P)}
            if world == 1:
                # the same keyframe through the device-resident map (SURVEY 8(f).2): the three keyframe clouds of the map frame are
                # already in HBM (Mapping::ToWorld put them there when their keyframes were registered); per keyframe: BuildMapFrame
                # (merge + voxel hash on the device), scan upload + scan-to-map, ToWorld of the new keyframe, eviction of the oldest
                fr = backend.FeatureAssociation(ctx)
                ident = np.array([0, 0, 0, 1, 0, 0, 0.0])
                thirds = np.array_split(np.arange(ICP_P), 3)
                for k, idx in enumerate(thirds):
                    fr.map_append(k, np.ascontiguousarray(sc["map"][idx]), ident)

                def keyframe():
                    fr.map_build([0, 1, 2], sc["cell_size"])
                    fr.scan_to_map(*argsicp)
                    fr.map_append(3, None, sc["frame_pose"])
                    fr.map_evict(3)
                for _ in range(3):
                    keyframe()
                walls = []
                for _ in range(5):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    keyframe()
                    torch.cuda.synchronize()
                    walls.append((time.perf_counter() - t0) * 1e3)
                line["icp"]["e2e_resident_map"] = {"value": ICP_K / (float(np.median(walls)) * 1e-3), "unit": "points/s", "ms_per_keyframe": float(np.median(walls)),
                                                   "note": "lvb_icp_map_build (3 resident keyframe clouds -> 1M-point map frame, on the device) + scan upload + "
                                                           "association + 4 LM iterations + lvb_icp_map_append of the registered scan + evict; host wall clock"}
                fr.close()
            isplit = kernel_split(lvb, lambda: fa.scan_to_map(*argsicp), 1)
            line["kernels"]["icp_us_per_scan"] = {k: round(v, 1) for k, v in sorted(isplit.items(), key=lambda kv: -kv[1])}
            us = isplit.get("icp_associate_kernel")
            if us and world == 1:
                alg = ICP_K * BYTES_KNN_QUERY + ICP_P * 16
                line["icp"]["knn_only"] = {"value": ICP_K / (us * 1e-6), "unit": "points/s", "us": us,
                                           "note": "icp_associate_kernel alone: float32 transform + exact 3-NN + gate + plane normal"}
                line["icp"]["roofline"] = {"bound": "hbm", "achieved": alg / (us * 1e-6) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / (us * 1e-6) / 1e9 / peak,
                                           "traffic": 17.53e6, "traffic_source": "profiles/icp_r2_final_summary.txt (ncu --set full), not measured in-run",
                                           "kernel": "icp_associate_kernel", "bytes_per_query": BYTES_KNN_QUERY + 16.0 * ICP_P / ICP_K,
                                           "us_per_launch": us, "peak_source": peak_src,
                                           "note": "algorithmic minimum of SURVEY 8(d) (40 B/query + the map read once); the voxel ring scan is L2-latency work on top"}

        # ---------------- lidar feature pipeline (SURVEY 8(f).2): raw 64 x 1800 sweep -> ground / surf features, host buffers in and out
        sweep = None
        if rank == 0 and not args.skip_icp:
            sweep = synth.make_lidar_scan(seed=synth.SEED)
            lf = backend.LidarFeatures(ctx1)
            for _ in range(3):
                gcl, scl = lf.extract(sweep)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(10):
                lf.extract(sweep)
            lf_ms = (time.perf_counter() - t0) * 1e3 / 10
            line["lidar_features"] = {"metric": "lidar_raw_points_per_s", "value": len(sweep) / (lf_ms * 1e-3), "unit": "points/s", "ms_per_sweep": lf_ms,
                                      "ground_points": int(len(gcl)), "surf_points": int(len(scl)),
                                      "workload": "FeatureAssociation::Process on a synthetic %d-point sweep (64 x 1800), e2e with H2D/D2H" % len(sweep)}

        sampler.join(timeout=2)
        line["clocks"] = sampler.summary()
        line["clocks"]["note"] = "sampled with nvidia-smi during the timed headline leg"

        # ---------------- CPU baseline beside it (rank 0, bounded samples)
        if rank == 0 and not args.skip_cpu:
            from oracle import binding
            orc = binding.load()
            T = cpu_threads()
            octx = backend.Context(orc)
            v10, it10, _ = cpu_window(orc, octx, N_KF, N_LM, 40, T)
            line["cpu_baseline"] = {"value": v10, "unit": "rows/s", "cores": T, "kind": "port",
                                    "sample": "%d LM iterations of the configs[1] window on the oracle restatement (%d threads of %d cores)" % (it10, T, os.cpu_count() or 1)}
            if "window20" in line:
                v20, it20, _ = cpu_window(orc, octx, W20_KF, W20_LM, 20, T)
                line["window20"]["cpu_baseline"] = {"value": v20, "unit": "rows/s", "cores": T, "kind": "port", "sample": "%d LM iterations of the same window" % it20}
                line["window20"]["vs_cpu"] = {"resident": line["window20"]["value"] / v20, "e2e": line["window20"]["e2e"]["value"] / v20}
            if "icp" in line and world == 1:
                line["icp"]["cpu_baseline"] = cpu_icp(orc, octx, T)
                line["icp"]["vs_cpu"] = {"resident": line["icp"]["value"] / line["icp"]["cpu_baseline"]["value"],
                                         "e2e": line["icp"]["e2e"]["value"] / line["icp"]["cpu_baseline"]["value"]}
            # the roofline kernel's CPU counterpart: the reference's own TwoFrameReprojectionError under forward-mode duals (what Ceres'
            # AutoDiff does per residual block), prebuilt where the reference tree is mounted (oracle/ref_time_harness.cpp); one thread, ~2 s
            ref_time = os.path.join(ROOT, "oracle", "_ref", "ref_time")
            if os.path.exists(ref_time):
                try:
                    t = subprocess.run([ref_time, "20000", "2.0"], capture_output=True, text=True, timeout=60, check=True).stdout.split()
                    line["cpu_baseline"]["eval_kernel"] = {"value": 2.0 * float(t[2]), "unit": "rows/s", "cores": 1, "kind": "reference",
                                                           "sample": "%s TwoFrameReprojectionError blocks (visual_error.hpp:78-107 compiled in place, residual + 2x15 Jacobian by duals) in %s s" % (t[0], t[1])}
                except Exception as exc:                      # a baseline beside the number, never a reason to lose the line
                    line["cpu_baseline"]["eval_kernel"] = {"unavailable": str(exc)[:120]}
            if "lidar_features" in line:
                olf = backend.LidarFeatures(octx)
                t0 = time.perf_counter()
                for _ in range(5):
                    olf.extract(sweep)
                line["lidar_features"]["cpu_port_points_per_s"] = len(sweep) / ((time.perf_counter() - t0) / 5)
        if rank == 0:
            print(json.dumps(line))
    if world > 1:
        dist.barrier()                  # rank 0 is still timing the CPU baseline: nobody tears the process group down under it
        torch.cuda.synchronize()
        ctx.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
