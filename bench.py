#!/usr/bin/env python
"""bench.py — point-associations/s of the LIO scan-matching hot path (BASELINE.json metric).

Workload (BASELINE config 2, `configs[1]`): 100k-pt Livox-pattern sweep vs a ~10M-pt voxel map, 3 ESIKF passes per
sweep, r3live.yaml parameters with the residual cap lifted (max_num_residuals >= N) and early convergence disabled so
that every step runs exactly 3 passes.  A "step" is one sweep = updateIEKF (3 x [fused K1 pass + 256-byte result +
17x17 host update]).  --gpus N shards the same sweep by point index over N ranks (config 3, strong scaling) with one
32-double all-reduce per pass.

  value : associations/s with the sweep already resident in HBM (C-ABI srl_update_iekf / sharded loop)
  e2e   : the same through the host-buffer entry point (srl_optimize_host: H2D of the sweep, passes, final
          re-transform, D2H of the registered points)
  --impl reference : the reference's own sources compiled where they lie (oracle/_ref/libsrl_reference.so) on all host
          threads, one independent sweep per thread; the oracle port when that library is absent — the reference arm.
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

METRIC = "point-associations/sec per ESIKF iter, 100k-pt sweep vs 10M-pt map"
UNIT = "associations/s"
BIG = 2 ** 31 - 1
N_PASSES = 3   # overridden by --passes


def bench_params(mod):
    # 3 passes exactly: i = -1, 0, 1 (num_iters_icp = 2), never "converged" early
    return mod.r3live_params(max_num_residuals=BIG, num_iters_icp=N_PASSES - 1, threshold_translation_norm=0.0,
                             threshold_orientation_norm=0.0, frame_id=100)


def make_sweeps(synth, n_points, n_sweeps, pattern="livox"):
    out = []
    for i in range(n_sweeps):
        pos = (40.0 * ((i % 5) - 2), 3.0 + 40.0 * ((i // 5) % 3 - 1), 1.8)
        out.append(synth.make_sweep(n_points, seed=1000 + i, yaw=0.5 + 0.37 * i, position=pos, pattern=pattern))
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, device_index=0):
        self.lines = []
        self.proc = None
        self.idx = device_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def run_reference(args):
    """CPU arm, wall-clock timed on rank 0.

    Default: the REFERENCE'S OWN CODE — oracle/_ref/libsrl_reference.so, /root/reference/src/optimize.cpp etc. compiled unmodified
    where they lie (oracle/Makefile) — on all host threads.  The reference has no threading on this path, so the only way it
    can use more than one core is independent sweeps: a step is one batch of `cores` sweeps, each registered against the shared
    map by its own thread through the reference's single-threaded updateIEKF (ref_update_iekf_many).  Each sweep is a bounded
    sample (a prefix of the random-order keypoints of a config-2 sweep) sized so that the whole run ends within a few minutes.
    Fallback (library not built, or SRL_CPU_ARM=port): the oracle port with keypoint ranges over std::threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle_py as O
    from oracle import reference_py as Rf
    from sr_livo_b200 import synth
    cores = os.cpu_count() or 1
    use_ref = Rf.available() and os.environ.get("SRL_CPU_ARM", "reference") != "port"
    prm = bench_params(O)
    P = synth.prior_covariance()
    sweeps = make_sweeps(synth, args.points, 8, args.pattern)
    if args.map_extent < 400.0:   # reduced maps (tests): keep the sensor positions that lie well inside the map
        sweeps = [sw for sw in sweeps if max(abs(sw.t_true[0]), abs(sw.t_true[1])) <= args.map_extent / 2.0 - 30.0] or sweeps[:1]
    t0 = time.time()
    pts = synth.sample_map_points(args.map_extent, 60.0, seed=1)
    om = O.OracleMap()
    om.add_points(pts)
    n_pts, n_vox = om.num_points, om.num_voxels
    del pts
    if use_ref:
        # the map is built once, by the port's addPointsToMap (8 s instead of 45 s for the 32 M offered points), and copied into
        # the reference's own voxelHashMap; tests/test_reference_pin.py shows both insertions give the same container content
        ref = Rf.Reference()
        keys, counts, xyz = om.snapshot()
        ref.load(keys, counts, xyz)
        del keys, counts, xyz
        assert ref.num_points() == n_pts and ref.num_voxels() == n_vox
    t_map = time.time() - t0
    extra = {}
    if use_ref:
        n_s = min(args.points, 25000)

        def batch(n_keypoints, first):
            # every thread registers its own slice of keypoints of ONE sweep (consecutive sweeps of a 10 Hz stream come from
            # almost the same place: the threads then share the map region in the caches, as the port's keypoint ranges do)
            sw = sweeps[first % len(sweeps)]
            n_slices = max(1, sw.raw_xyz.shape[0] // n_keypoints)
            raws = [sw.raw_xyz[(j % n_slices) * n_keypoints:(j % n_slices + 1) * n_keypoints] for j in range(cores)]
            es = [O.Eskf(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=P.copy()) for j in range(cores)]
            tls = [sw.t_last] * cores
            t = time.perf_counter()
            ok, out, fq, ft = ref.update_iekf_many(raws, es, tls, prm, n_threads=cores)
            dt = time.perf_counter() - t
            assert ok == cores, (ok, cores)
            return dt, out, [first % len(sweeps)]
        t_probe = batch(n_s, 0)[0]                               # first warm-up batch, also sizes the sample:
        budget_s = 45.0                                           # all warm-up + timed batches together stay near this
        if (args.steps + args.warmup) * t_probe > budget_s:
            n_s = max(2000, int(n_s * budget_s / ((args.steps + args.warmup) * t_probe)) // 32 * 32)
        for i in range(1, max(args.warmup, 1)):
            batch(n_s, i)
        ts = []
        for i in range(args.steps):
            dt_i, out, idx = batch(n_s, args.warmup + i)
            ts.append(dt_i)
        dt = float(np.sum(ts)) / max(args.steps, 1)
        units = cores * n_s * N_PASSES
        value = units / dt
        # single thread = the reference exactly as written (one sweep, one core), and a cross-check of one result against the port
        t = time.perf_counter()
        one = ref.update_iekf(sweeps[idx[0]].raw_xyz[:n_s], O.Eskf(p=sweeps[idx[0]].t_init.copy(), q=sweeps[idx[0]].q_init.copy(), cov=P.copy()),
                              sweeps[idx[0]].t_last, prm)
        t_one = time.perf_counter() - t
        po = om.update_iekf(sweeps[idx[0]].raw_xyz[:n_s], O.Eskf(p=sweeps[idx[0]].t_init.copy(), q=sweeps[idx[0]].q_init.copy(), cov=P.copy()),
                            sweeps[idx[0]].t_last, prm, nthreads=cores)
        assert po["passes"] == N_PASSES, po["passes"]
        # the oracle port on the same host: whole sweeps, keypoint ranges over all threads (the other way to use every core)
        t_ports = []
        for i in range(max(3, min(args.steps, 20))):
            sw = sweeps[(args.warmup + i) % len(sweeps)]
            t = time.perf_counter()
            om.update_iekf(sw.raw_xyz, O.Eskf(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=P.copy()), sw.t_last, prm, nthreads=cores)
            t_ports.append(time.perf_counter() - t)
        port_value = args.points * N_PASSES / (float(np.sum(t_ports[1:])) / (len(t_ports) - 1))
        ref_value = value
        kind = "reference"
        sample = (f"{args.steps} batches x {cores} independent sweeps ({n_s}-keypoint slices of one {args.points}-pt sweep per batch) x {N_PASSES} passes, "
                  f"one sweep per host thread through the reference's own single-threaded updateIEKF, shared map")
        if port_value > ref_value:
            # report the stronger CPU number: a ratio against the weaker one would flatter the GPU
            value, dt, kind = port_value, args.points * N_PASSES / port_value, "port"
            sample = (f"the oracle port was the faster CPU form on this host: whole {args.points}-keypoint sweeps x {N_PASSES} passes, keypoint ranges over "
                      f"{cores} std::threads, {len(t_ports) - 1} sweeps; reference_value = " + sample)
        extra = {"reference_value": ref_value, "port_value": port_value, "single_thread_value": n_s * N_PASSES / t_one,
                 "pose_equals_port": bool(np.allclose(out[0].p, po["eskf"].p, rtol=0, atol=1e-9) and np.allclose(one["eskf"].p, po["eskf"].p, rtol=0, atol=1e-9)),
                 "library": Rf.lib().ref_build_info().decode()}
        container = "tsl::robin_map 0.6.3 (reference vendored header), the reference's own voxelHashMap"
        workload_note = (f"; sample: {n_s}-keypoint slices of one sweep, one per host thread" if kind == "reference"
                         else "; whole sweeps, keypoint ranges over the host threads (faster than the compiled reference's one-sweep-per-thread form here)")
    else:
        def step(sw):
            e = O.Eskf(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=P.copy())
            r = om.update_iekf(sw.raw_xyz, e, sw.t_last, prm, nthreads=cores)
            assert r["passes"] == N_PASSES, r["passes"]
            return r
        for i in range(args.warmup):
            step(sweeps[i % len(sweeps)])
        t0 = time.perf_counter()
        for i in range(args.steps):
            step(sweeps[(args.warmup + i) % len(sweeps)])
        dt = (time.perf_counter() - t0) / max(args.steps, 1)
        value = args.points * N_PASSES / dt
        kind = "port"   # restated algorithm (oracle/srl_oracle.cpp) over the reference's robin-map
        sample = (f"whole workload: {args.steps} sweeps x {N_PASSES} passes x {args.points} keypoints, keypoint ranges over {cores} std::threads")
        container = O.backend()
        workload_note = ""
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"cfg2: {args.points}-pt {args.pattern} sweep vs {n_pts}-pt map ({n_vox} voxels), "
                                   f"{N_PASSES} ESIKF passes/step, r3live params, cap lifted", "container": container,
                       "map_build_s": round(t_map, 1), "cpu_arm": kind + workload_note},
            "cpu_baseline": dict({"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample}, **extra),
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)
    return 0


def run_cfg5(args, torch, tdist, dist, lio, synth, rank, world, local, stream, flush_buf, peak):
    """BASELINE configs[4]: 500k-pt dense spinning-LiDAR sweep, ~50M-pt map, 5 ESIKF passes, sharded over `world` GPUs.
    Same timing rules as the main workload (events per step, L2 flush between steps, max over ranks)."""
    n_pts5, passes5, steps5, warm5 = 500000, 5, args.cfg5_steps, 3
    dev = f"cuda:{local}"
    L5 = lio.LioOptimization(device=local, stream=stream, max_voxels=1 << 23, sweep_capacity=n_pts5)
    # rank 0 samples the world (~156M offered points, ~40 s of numpy); the others receive it over NVLink
    t0 = time.time()
    if rank == 0:
        pts = synth.sample_map_points(1340.0, 60.0, seed=1)
        n_off = torch.tensor([pts.shape[0]], dtype=torch.int64, device=dev)
    else:
        pts = None
        n_off = torch.zeros(1, dtype=torch.int64, device=dev)
    if world > 1:
        tdist.broadcast(n_off, src=0)
    d_pts = torch.empty((int(n_off.item()), 3), dtype=torch.float64, device=dev)
    if rank == 0:
        d_pts.copy_(torch.from_numpy(pts))
        del pts
    if world > 1:
        tdist.broadcast(d_pts, src=0)
    torch.cuda.synchronize()
    t_gen = time.time() - t0
    t0 = time.time()
    L5.voxel_map.insert_device(d_pts.data_ptr(), d_pts.shape[0])
    t_ins = time.time() - t0
    del d_pts
    torch.cuda.empty_cache()
    n_vox, n_map = L5.voxel_map.stats()
    sweeps = make_sweeps(synth, n_pts5, 2, "spinning")
    prm = lio.r3live_params(max_num_residuals=BIG, num_iters_icp=passes5 - 1, threshold_translation_norm=0.0,
                            threshold_orientation_norm=0.0, frame_id=100)
    P = synth.prior_covariance()
    d_raw = [torch.from_numpy(s.raw_xyz).to(dev) for s in sweeps]
    D5 = dist.DistributedLio(L5, rank, world, native=True) if world > 1 else None
    pin_world = torch.empty((n_pts5, 3), dtype=torch.float64).pin_memory()
    world_out = pin_world.numpy()
    pin_raw = [torch.from_numpy(s.raw_xyz).pin_memory() for s in sweeps]

    def prepare(i):
        sw = sweeps[i % len(sweeps)]
        if world > 1:
            D5.set_keypoints_device(d_raw[i % len(sweeps)].data_ptr(), n_pts5)
        else:
            L5.sweep.set_device(d_raw[i % len(sweeps)].data_ptr(), n_pts5)
        L5.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=P.copy())
        return sw

    def step_resident(i, sw):
        if world > 1:
            out = D5.updateIEKF(prm, sw.t_last)
            assert out["success"] and out["passes"] == passes5, out["passes"]
        else:
            summ, _, _ = L5.updateIEKF(prm, sw.t_last)
            assert summ.success and summ.passes_run == passes5

    def step_e2e(i, sw):
        L5.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=P.copy())
        raw_h = pin_raw[i % len(sweeps)].numpy()
        if world > 1:
            out = D5.optimize(raw_h, prm, sw.t_last, world_out=world_out)
            assert out["success"] and out["passes"] == passes5
        else:
            summ, _, _, _ = L5.optimize(raw_h, prm, sw.t_last, want_world=True, world_out=world_out)
            assert summ.success and summ.passes_run == passes5

    def barrier():
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, with_prepare):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps5)]
        for i in range(warm5):
            step_fn(i, prepare(i) if with_prepare else sweeps[i % len(sweeps)])
        L5.ctx.pass_time(reset=True)
        barrier()
        for i in range(steps5):
            sw = prepare(warm5 + i) if with_prepare else sweeps[(warm5 + i) % len(sweeps)]
            flush_buf.fill_(i & 0xff)
            if world > 1:
                tdist.barrier()
            ev[i][0].record()
            step_fn(warm5 + i, sw)
            ev[i][1].record()
        barrier()
        ms = np.array([a.elapsed_time(b) for a, b in ev])
        k1_ms, k1_n = L5.ctx.pass_time(reset=True)
        return ms, k1_ms, k1_n

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            tdist.all_reduce(t, op=tdist.ReduceOp.SUM)
        return float(t.item())
    ms_res, _, _ = timed(step_resident, True)
    ms_e2e, _, _ = timed(step_e2e, False)
    L5.ctx.set_timing(True)
    _, k1_ms, k1_n = timed(step_resident, True)
    L5.ctx.set_timing(False)
    ms_step, ms_step_e2e = max_over_ranks(float(ms_res.mean())), max_over_ranks(float(ms_e2e.mean()))
    k1_avg = max_over_ranks(k1_ms / max(k1_n, 1))
    # algorithmic bytes of one pass over the whole sweep: 456 N + 12 * (candidates the GPU scanned, summed over ranks)
    sw0 = prepare(0)
    gp = L5.buildPlaneResiduals(prm, sw0.q_init, sw0.t_init, sw0.t_last)
    scanned = sum_over_ranks(float(gp.num_candidates_scanned))
    alg_bytes = 456.0 * n_pts5 + 12.0 * scanned
    out = {"workload": f"cfg5: {n_pts5}-pt spinning sweep vs {n_map}-pt map ({n_vox} voxels), {passes5} ESIKF passes/step, "
                       f"r3live params, cap lifted, {world} GPU(s)",
           "value": n_pts5 * passes5 / (ms_step * 1e-3), "unit": UNIT, "ms_per_step": ms_step, "steps": steps5, "warmup": warm5,
           "e2e": {"value": n_pts5 * passes5 / (ms_step_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_step_e2e,
                   "h2d_bytes_per_step": n_pts5 * 24, "d2h_bytes_per_step": n_pts5 * 24 + world * 9328},
           "roofline": {"bound": "hbm", "achieved": alg_bytes / world / (k1_avg * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": alg_bytes / world / (k1_avg * 1e-3) / 1e9 / peak, "bytes_per_launch_per_gpu": alg_bytes / world,
                        "bytes_basis": "GPU-scanned candidates, summed over ranks (the oracle's sum C_k is an N=1 leg)",
                        "k1_avg_ms": k1_avg, "note": "per-GPU achieved bandwidth of one pass (incl. the wait for the pose ticket)"},
           "ms_per_step_stats": {"resident": {"p50": float(np.median(ms_res)), "min": float(ms_res.min()), "max": float(ms_res.max())},
                                 "e2e": {"p50": float(np.median(ms_e2e)), "min": float(ms_e2e.min()), "max": float(ms_e2e.max())},
                                 "note": "this rank's per-step CUDA-event times; the values above are their means (max over ranks)"},
           "map_gen_s": round(t_gen, 1), "map_insert_s": round(t_ins, 2)}
    if D5 is not None:
        D5.close()
    L5.close()
    return out


def step_outputs(leg, last, eskf):
    """What a caller of the timed path receives from one step: the registered pose, the filter state and the pass summary.
    `last` is (summary, frame_q, frame_t) on one GPU, the result dict of DistributedLio on several."""
    if isinstance(last, dict):
        fq, ft = last["frame_q"], last["frame_t"]
        summary, trace = [last["success"], last["passes"], last["num_residuals_used"], last["converged"]], last["trace"]
    else:
        s, fq, ft = last
        summary, trace = [s.success, s.passes_run, s.num_residuals_used, s.converged], s.trace
    out = {f"{leg}_frame_q": fq, f"{leg}_frame_t": ft, f"{leg}_summary": summary, f"{leg}_trace": trace,
           **{f"{leg}_{f}": getattr(eskf, f) for f in ("p", "q", "v", "ba", "bg", "g", "cov")}}
    return out


def dump_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), np.asarray(a, dtype=np.float64))


_REAL_STDOUT = None


def emit(line):
    """The one JSON line of the contract goes to the process's real stdout; everything else a library prints to fd 1
    during the run (e.g. NCCL's version banner) was rerouted to stderr by main()."""
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--points", type=int, default=100000)
    ap.add_argument("--map-extent", type=float, default=600.0, help="side of the square world in m (600 -> ~10M points)")
    ap.add_argument("--passes", type=int, default=3, help="ESIKF passes per sweep (config 2: 3, config 5: 5)")
    ap.add_argument("--pattern", default="livox", choices=["livox", "spinning"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--k1-variant", type=int, default=0, help="0 auto, 1 k1_fast, 2 k1_assoc only, 3 k1_scan + k1_fit (A/B runs)")
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between timed steps")
    ap.add_argument("--cfg5", action="store_true", help="also run the config-5 block (500k-pt spinning sweep, ~50M-pt map, 5 passes); "
                                                        "on by default when --gpus > 1")
    ap.add_argument("--no-cfg5", action="store_true")
    ap.add_argument("--cfg5-steps", type=int, default=10)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (float64), "
                                                           "so that two builds can be compared output for output")
    args = ap.parse_args()
    global N_PASSES
    N_PASSES = args.passes
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the outputs of the GPU path (--impl b200)")
        return run_reference(args)

    import torch
    import torch.distributed as tdist
    from sr_livo_b200 import dist, lio, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the scan-matching path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        tdist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(f"cuda:{local}"))
    stream = torch.cuda.current_stream().cuda_stream or 1        # 1 == cudaStreamLegacy
    L = lio.LioOptimization(device=local, stream=stream, max_voxels=1 << 21 if args.map_extent <= 900 else 1 << 23,
                            sweep_capacity=max(args.points, 1024))
    if args.k1_variant:
        L.ctx.set_option("k1_variant", args.k1_variant)

    # ---- map: built by the product's own insert kernel (every rank builds its replica from the same seed)
    t0 = time.time()
    pts = synth.sample_map_points(args.map_extent, 60.0, seed=1)
    t_gen = time.time() - t0
    t0 = time.time()
    L.addPointsToMap(pts)
    t_ins = time.time() - t0
    n_offered = pts.shape[0]
    del pts
    n_vox, n_pts = L.voxel_map.stats()
    sweeps = make_sweeps(synth, args.points, 8, args.pattern)
    prm = bench_params(lio)
    P = synth.prior_covariance()
    d_raw = [torch.from_numpy(s.raw_xyz).to(f"cuda:{local}") for s in sweeps]
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=f"cuda:{local}")   # > 126 MB L2
    native = os.environ.get("SRL_DIST_NATIVE", "1") != "0"
    D = dist.DistributedLio(L, rank, world, native=native) if world > 1 else None

    def prepare(i):
        sw = sweeps[i % len(sweeps)]
        if world > 1:
            D.set_keypoints_device(d_raw[i % len(sweeps)].data_ptr(), sw.raw_xyz.shape[0])   # this rank's range only
        else:
            L.sweep.set_device(d_raw[i % len(sweeps)].data_ptr(), sw.raw_xyz.shape[0])
        L.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=P.copy())
        return sw

    def step_resident(sw):
        if world > 1:
            out = D.updateIEKF(prm, sw.t_last)
            assert out["success"] and out["passes"] == N_PASSES
            return out
        summ, fq, ft = L.updateIEKF(prm, sw.t_last)
        assert summ.success and summ.passes_run == N_PASSES, (summ.success, summ.passes_run)
        return summ, fq, ft

    # e2e leg: the host buffers a caller would hand over, in pinned memory (the contract's "from pinned host memory")
    pin_world = torch.empty((args.points, 3), dtype=torch.float64).pin_memory()
    world_out = pin_world.numpy()
    pin_raw = [torch.from_numpy(s.raw_xyz).pin_memory() for s in sweeps]
    raw_host = {id(s): t.numpy() for s, t in zip(sweeps, pin_raw)}

    def step_e2e(sw):
        L.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=P.copy())
        raw_h = raw_host[id(sw)]
        if world > 1:
            out = D.optimize(raw_h, prm, sw.t_last, world_out=world_out)   # srl_optimize_host_dist: all in C, pinned buffers
            assert out["success"] and out["passes"] == N_PASSES
            return out
        summ, fq, ft, w = L.optimize(raw_h, prm, sw.t_last, want_world=True, world_out=world_out)
        assert summ.success and summ.passes_run == N_PASSES
        return summ, fq, ft

    def barrier():
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, with_prepare, n_steps=None):
        n_steps = args.steps if n_steps is None else n_steps
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_steps)]
        for i in range(args.warmup):
            sw = prepare(i) if with_prepare else sweeps[i % len(sweeps)]
            step_fn(sw)
        L.ctx.pass_time(reset=True)
        launches0 = L.ctx.kernel_launches
        barrier()
        last = None
        for i in range(n_steps):
            sw = prepare(args.warmup + i) if with_prepare else sweeps[(args.warmup + i) % len(sweeps)]
            if not args.no_flush:
                flush_buf.fill_(i & 0xff)                                  # evict L2 between timed steps (untimed)
            if world > 1:
                tdist.barrier()
            ev[i][0].record()
            last = step_fn(sw)
            ev[i][1].record()
        barrier()
        ms = np.array([a.elapsed_time(b) for a, b in ev])
        k1_ms, k1_n = L.ctx.pass_time(reset=True)
        return ms, k1_ms, k1_n, L.ctx.kernel_launches - launches0, last

    clocks = ClockSampler(local)
    clocks.start()
    ms_res, _, _, launches, last_res = timed(step_resident, True)
    outputs = step_outputs("resident", last_res, L.eskf_pro) if args.dump_outputs else None
    step_cycles = L.ctx.counter("iekf_step_cycles_avg")
    loop_on_device = bool(L.ctx.counter("device_loop_active"))
    order_impl = {1: "single-launch cluster radix sort (k_sweep_order_cluster), verified against the CUB order at first use",
                  0: "CUB radix sort", -1: "cluster radix sort, still in its first verified uses"}.get(L.ctx.counter("cluster_order_active"), "?")
    stage_cycles = [L.ctx.counter(f"iekf_stage_{i}") for i in range(8)]
    ms_e2e, _, _, _, last_e2e = timed(step_e2e, False)
    if outputs is not None:
        outputs.update(step_outputs("e2e", last_e2e, L.eskf_pro), e2e_world=world_out.copy())
    # roofline leg: the same resident steps again with CUDA events around every pass's launches on the launching stream
    # (the events sit between the kernels, so this leg runs without programmatic dependent launch; its step time is
    # reported next to the main one)
    L.ctx.set_timing(True)
    ms_tim, k1_ms, k1_n, _, _ = timed(step_resident, True, n_steps=min(args.steps, 40))
    L.ctx.set_timing(False)
    clk = clocks.stop()   # sampled over the three timed regions

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
        if world > 1:
            tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
        return float(t.item())
    ms_step = max_over_ranks(float(ms_res.mean()))
    ms_step_e2e = max_over_ranks(float(ms_e2e.mean()))
    ms_step_tim = max_over_ranks(float(ms_tim.mean()))
    k1_avg_ms = max_over_ranks(k1_ms / max(k1_n, 1))
    value = args.points * N_PASSES / (ms_step * 1e-3)
    e2e_value = args.points * N_PASSES / (ms_step_e2e * 1e-3)

    # ---- roofline of the pass (k1_scan dominant): algorithmic bytes / measured duration of the pass's launches
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"]); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak = 6650.0; peak_src = "fallback 6.65 TB/s (B200_PROFILING.md)"
    sw0 = sweeps[0]
    n_shard = args.points if world == 1 else (dist.shard_range(args.points, rank, world)[1] - dist.shard_range(args.points, rank, world)[0])
    prepare(0)
    gp = L.buildPlaneResiduals(prm, sw0.q_init, sw0.t_init, sw0.t_last)
    bytes_gpu_scanned = 456.0 * n_shard + 12.0 * gp.num_candidates_scanned

    cpu_baseline = None
    sumC = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle_py as O                                  # the one place bench.py runs the oracle
        cores = os.cpu_count() or 1
        keys, counts, xyz = L.voxel_map.download()
        om = O.OracleMap()
        om.load(keys, counts, xyz)
        oprm = bench_params(O)
        o1 = om.build_plane_residuals(sw0.raw_xyz, sw0.q_init, sw0.t_init, sw0.t_last, oprm, nthreads=cores)
        sumC = int(o1.sum_candidates)
        rel = float(np.abs(o1.HTH - gp.HTH).max() / np.abs(o1.HTH).max())
        ts = []
        for rep in range(3):
            t0 = time.perf_counter()
            r = om.update_iekf(sw0.raw_xyz, O.Eskf(p=sw0.t_init.copy(), q=sw0.q_init.copy(), cov=P.copy()), sw0.t_last, oprm, nthreads=cores)
            ts.append(time.perf_counter() - t0)
        t_all = float(np.median(ts))
        n1 = min(args.points, 20000)
        t0 = time.perf_counter()
        om.update_iekf(sw0.raw_xyz[:n1], O.Eskf(p=sw0.t_init.copy(), q=sw0.q_init.copy(), cov=P.copy()), sw0.t_last, oprm, nthreads=1)
        t_one = time.perf_counter() - t0
        cpu_baseline = {"value": args.points * N_PASSES / t_all, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": f"one sweep ({args.points} keypoints x {N_PASSES} passes), median of 3, {cores} std::threads; "
                                  f"single-thread (reference as written) on {n1} keypoints x {N_PASSES} passes",
                        "single_thread_value": n1 * N_PASSES / t_one, "container": O.backend(),
                        "pass_parity_HTH_rel": rel, "residuals_equal": bool(o1.num_residuals == gp.num_residuals)}
        # the reference's own sources compiled where they lie (oracle/_ref/libsrl_reference.so), when that library travelled here:
        # one independent sweep per host thread (the reference is single-threaded on this path), a bounded sample of n1 keypoints each
        try:
            from oracle import reference_py as Rf
            if Rf.available() and os.environ.get("SRL_CPU_ARM", "reference") != "port":
                ref = Rf.Reference()
                ref.load(keys, counts, xyz)
                n_slices = max(1, sw0.raw_xyz.shape[0] // n1)             # every thread its own keypoint slice of the same sweep
                raws = [sw0.raw_xyz[(j % n_slices) * n1:(j % n_slices + 1) * n1] for j in range(cores)]
                tls = [sw0.t_last] * cores
                t_many = []
                for rep in range(2):
                    es = [O.Eskf(p=sw0.t_init.copy(), q=sw0.q_init.copy(), cov=P.copy()) for j in range(cores)]
                    t0 = time.perf_counter()
                    ok, out, _, _ = ref.update_iekf_many(raws, es, tls, oprm, n_threads=cores)
                    t_many.append(time.perf_counter() - t0)
                t0 = time.perf_counter()
                one = ref.update_iekf(sw0.raw_xyz[:n1], O.Eskf(p=sw0.t_init.copy(), q=sw0.q_init.copy(), cov=P.copy()), sw0.t_last, oprm)
                t_ref_one = time.perf_counter() - t0
                po = om.update_iekf(sw0.raw_xyz[:n1], O.Eskf(p=sw0.t_init.copy(), q=sw0.q_init.copy(), cov=P.copy()), sw0.t_last, oprm, nthreads=cores)
                if ok == cores:
                    ref_value = cores * n1 * N_PASSES / min(t_many)
                    cpu_baseline.update({
                        "port_value": cpu_baseline["value"], "port_single_thread_value": cpu_baseline["single_thread_value"],
                        "reference_value": ref_value, "reference_single_thread_value": n1 * N_PASSES / t_ref_one,
                        "pose_equals_port": bool(np.allclose(one["eskf"].p, po["eskf"].p, rtol=0, atol=1e-9)),
                        "sample": cpu_baseline["sample"] + f"; reference_*: the reference's own sources (oracle/_ref/libsrl_reference.so), {cores} independent "
                                  f"sweeps ({n1}-keypoint slices of the same sweep) x {N_PASSES} passes, one per host thread through its single-threaded "
                                  f"updateIEKF, shared map, best of 2; value = the faster of the two CPU forms"})
                    if ref_value > cpu_baseline["value"]:
                        cpu_baseline.update({"value": ref_value, "kind": "reference", "single_thread_value": n1 * N_PASSES / t_ref_one})
                del ref
        except Exception as ex:   # the port numbers above stand
            cpu_baseline["reference_library_error"] = repr(ex)[:200]
    if sumC is not None:
        alg_bytes = 456.0 * n_shard + 12.0 * sumC
        basis = "reference-visited candidates (oracle sum C_k on sweep 0)"
    else:
        alg_bytes = bytes_gpu_scanned
        basis = "GPU-scanned candidates (oracle leg not run at this N)"
    achieved = alg_bytes / (k1_avg_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "one ESIKF pass = k1_scan + k1_fit + k1_assoc (exact fallback, usually empty); dominant: k1_scan", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "peak_source": peak_src, "bytes_per_launch": alg_bytes, "bytes_basis": basis,
                "bytes_gpu_scanned": bytes_gpu_scanned, "k1_avg_ms": k1_avg_ms, "k1_launches": int(k1_n),
                "k1_share_of_step": k1_avg_ms * N_PASSES / ms_step_tim, "timing_leg_ms_per_step": ms_step_tim,
                "note": "k1_avg_ms = CUDA events around each pass's launches (k1_scan incl. its wait for the pose ticket, k1_fit, "
                        "fallback), measured in a separate leg of the same resident steps"}
    tp = os.path.join(ROOT, "profiles", "k1_traffic.json")
    if os.path.exists(tp):
        try:
            roofline["traffic"] = json.load(open(tp)).get("dram_bytes_per_launch")
        except Exception:
            pass

    # ---- config 4 (extra, N=1 only): stream of sweeps, each registered (3 passes) and then inserted into the map
    streaming = None
    if world == 1:
        n_stream = 10
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
               for _ in range(n_stream)]
        added_total = 0
        for i in range(n_stream):
            sw = sweeps[i % len(sweeps)]
            evs[i][0].record()
            L.sweep.set_device(d_raw[i % len(sweeps)].data_ptr(), sw.raw_xyz.shape[0])
            L.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=P.copy())
            summ, fq, ft = L.updateIEKF(prm, sw.t_last)
            evs[i][1].record()
            added_total += L.addSweepToMap(fq, ft)
            evs[i][2].record()
        torch.cuda.synchronize()
        st_reg = np.array([a.elapsed_time(b) for a, b, c in evs])
        st_ins = np.array([b.elapsed_time(c) for a, b, c in evs])
        streaming = {"workload": f"cfg4: {n_stream} sweeps x ({N_PASSES} passes + map insert of the {args.points} registered points)",
                     "sweeps_per_s": 1e3 / float((st_reg + st_ins).mean()), "register_ms": float(st_reg.mean()),
                     "insert_ms": float(st_ins.mean()), "points_added_per_sweep": added_total / n_stream,
                     "realtime_factor_at_10hz": 100.0 / float((st_reg + st_ins).mean())}

    # ---- config 5 (extra block, default when N > 1): 500k-pt spinning sweep vs a ~50M-pt map, 5 passes, sharded over the ranks
    cfg5 = None
    if (world > 1 or args.cfg5) and not args.no_cfg5:
        cfg5 = run_cfg5(args, torch, tdist, dist, lio, synth, rank, world, local, stream, flush_buf, peak)

    # ---- N > 1: the sharded result must be the single-GPU result (sweep 0, whole sweep on this rank without the exchange)
    pose_check = None
    if world > 1:
        sw = prepare(0)
        out = D.updateIEKF(prm, sw.t_last)
        L.sweep.set_device(d_raw[0].data_ptr(), sw.raw_xyz.shape[0])
        L.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=P.copy())
        s1, q1, t1 = L.updateIEKF(prm, sw.t_last)
        dq = float(np.abs(np.asarray(out["frame_q"]) - q1).max()); dt = float(np.abs(np.asarray(out["frame_t"]) - t1).max())
        pose_check = {"sweep": 0, "max_abs_dq_vs_single_gpu": max_over_ranks(dq), "max_abs_dt_vs_single_gpu": max_over_ranks(dt),
                      "passes": [int(out["passes"]), int(s1.passes_run)]}
        assert pose_check["max_abs_dq_vs_single_gpu"] < 1e-8 and pose_check["max_abs_dt_vs_single_gpu"] < 1e-8, pose_check
        assert out["passes"] == s1.passes_run

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic",
                "config": {"workload": f"cfg{2 if world == 1 else 3}: {args.points}-pt {args.pattern} sweep vs {n_pts}-pt map ({n_vox} voxels), "
                                       f"{N_PASSES} ESIKF passes/step, r3live params, cap lifted",
                           "parallelism": (f"point-index shards x{world}, map replicated, 32 f64 per pass exchanged "
                                           + ("inside the pass's last kernel over NVLink peer memory (CUDA IPC mailboxes)" if native else
                                              "with one NCCL all-reduce")) if world > 1 else "single GPU",
                           "l2": "no flush" if args.no_flush else "256 MB L2 flush between timed steps; 8 distinct sweeps cycled",
                           "sweep_order": order_impl, "map_offered_points": int(n_offered), "map_gen_s": round(t_gen, 2), "map_insert_s": round(t_ins, 2)},
                "sweeps_per_s": 1e3 / ms_step, "clocks": clk, "gpu_launches": int(launches),
                "ms_per_step_stats": {"p50": float(np.median(ms_res)), "min": float(ms_res.min()), "max": float(ms_res.max()),
                                      "note": "this rank's per-step CUDA-event times; ms_per_step is their mean (max over ranks)"},
                "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_step_e2e,
                        "h2d_bytes_per_step": int(args.points * 24),
                        "d2h_bytes_per_step": int(args.points * 24 + (world * 9328 if loop_on_device else world * N_PASSES * 256)),
                        "entry_point": "srl_optimize_host_dist (C, pinned buffers, this rank's range only)" if world > 1 else "srl_optimize_host"},
                "roofline": roofline,
                "iekf_step": {"where": "device (persistent ESIKF block, srl_iekf.cu)" if loop_on_device else "host (srl_iekf_step)",
                              "sm_cycles_sums_to_pose": step_cycles,
                              "sm_cycles_to_stage": dict(zip(["-", "M", "inverse6", "d_x", "guard", "observe_quat", "observe_g", "post_jac"], stage_cycles))}}
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        if streaming is not None:
            line["streaming"] = streaming
        if cfg5 is not None:
            line["cfg5"] = cfg5
        if pose_check is not None:
            line["pose_check"] = pose_check
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        emit(line)
    if D is not None:
        D.close()
    if world > 1:
        tdist.destroy_process_group()
    L.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
