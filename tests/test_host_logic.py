"""CPU tests of the product's host side: the C-ABI library loads and exports every declared symbol, the host ESIKF
algebra (srl_iekf_step / srl_eskf_observe) agrees with the oracle, the host build of the per-keypoint math agrees
with numpy, and the point-index sharding + all-reduce loop works with world_size 2 over gloo.  No GPU compute here."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle_py as O
from oracle import reference_py as Rf
from refstore import Store, eskf_fields
from sr_livo_b200 import capi, dist, lio, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIG = 2 ** 31 - 1


@pytest.fixture(scope="module")
def ref_out():
    """outputs of the reference's own code (tests/refstore.py), stored in tests/golden/reference_host.npz"""
    store = Store("reference_host.npz")
    yield store
    store.save()


def test_library_exports_every_symbol_the_header_declares():
    hdr = open(os.path.join(ROOT, "include", "srlivo_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(srl_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(capi.EXPORTS), declared ^ set(capi.EXPORTS)
    L = capi.lib()
    for name in declared:
        assert hasattr(L, name), name
    assert L.srl_abi_version() == 1
    out = subprocess.run(["nm", "-D", "--defined-only", capi.LIB_PATH], capture_output=True, text=True).stdout
    for name in declared:
        assert re.search(rf"\bT {name}\b", out), f"{name} is not an exported text symbol"


def test_struct_layouts_match_the_header():
    # sizes the C compiler gives the structs (a mismatch here would silently corrupt every call)
    src = r'''
    #include <stdio.h>
    #include "srlivo_b200.h"
    int main(){ printf("%zu %zu %zu %zu %zu %zu %zu\n", sizeof(srl_icp_params), sizeof(srl_eskf_state), sizeof(srl_frame),
        sizeof(srl_normal_eq), sizeof(srl_debug_out), sizeof(srl_iekf_summary), sizeof(srl_iekf_iter)); return 0; }'''
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(d, "t"), os.path.join(d, "t.c")])
        sizes = [int(x) for x in subprocess.check_output([os.path.join(d, "t")]).split()]
    py = [C.sizeof(t) for t in (capi.IcpParams, capi.EskfState, capi.Frame, capi.NormalEq, capi.DebugOut,
                                capi.IekfSummary, capi.IekfIter)]
    assert sizes == py


def test_no_cpu_fallback_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    h = C.c_void_p()
    assert capi.lib().srl_ctx_create(0, None, C.byref(h)) == capi.SRL_CUDA_ERROR
    with pytest.raises(capi.SrlError):
        lio.Context(0)


def test_r3live_defaults_match_the_yaml():
    p = capi.r3live_params()
    o = O.r3live_params()
    for f, _ in capi.IcpParams._fields_:
        assert getattr(p, f) == getattr(o, f), f
    assert (p.size_voxel_map, p.num_iters_icp, p.min_number_neighbors, p.max_num_residuals) == (1.0, 5, 20, 600)


def test_eskf_observe_matches_oracle():
    rng = np.random.default_rng(3)
    for trial in range(20):
        scale = [0.05, 1e-6, 0.5][trial % 3]
        q = synth.quat_from_rotvec(rng.normal(size=3))
        kw = dict(p=rng.normal(size=3), q=q, v=rng.normal(size=3), ba=rng.normal(size=3) * 0.01,
                  bg=rng.normal(size=3) * 0.01, g=np.array([0.3, -0.2, 9.7]) + rng.normal(size=3) * 0.1)
        dx = rng.normal(size=17) * scale
        a = lio.EskfEstimator(**kw).observe(dx)
        b = O.Eskf(**kw).observe(dx)
        for f in ("p", "q", "v", "ba", "bg", "g"):
            assert np.allclose(getattr(a, f), getattr(b, f), rtol=0, atol=1e-14), f


def _run_product_host_loop(om, sw, oprm, prm, P):
    """The product's host algebra driven by ORACLE passes (so it runs without a GPU)."""
    st = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=P.copy()).to_c()
    fq, ft = sw.q_init.copy(), sw.t_init.copy()
    it = capi.IekfIter()
    assert capi.lib().srl_iekf_begin(C.byref(st), C.byref(prm), C.byref(it)) == 0
    trace = []
    while True:
        r = om.build_plane_residuals(sw.raw_xyz, fq, ft, sw.t_last, oprm)
        ne = capi.NormalEq()
        for i, v in enumerate(r.HTH.reshape(-1)):
            ne.HTH[i] = v
        for i, v in enumerate(r.HTh):
            ne.HTh[i] = v
        ne.num_residuals = r.num_residuals
        dx = np.zeros(17)
        done, div = C.c_int32(0), C.c_int32(0)
        rc = capi.lib().srl_iekf_step(C.byref(it), C.byref(ne), C.byref(prm), C.byref(st), capi.ptr(fq), capi.ptr(ft),
                                      capi.ptr(dx), C.byref(done), C.byref(div))
        assert rc == 0
        trace.append(np.concatenate([dx, ft, fq]))
        if done.value:
            break
    return lio.EskfEstimator.from_c(st), np.array(trace), done.value


@pytest.mark.parametrize("frame_id,thr_t", [(100, 0.01), (100, 0.0)])
def test_iekf_host_algebra_matches_oracle(small_world, frame_id, thr_t):
    om, sw = small_world["omap"], small_world["sweep"]
    kw = dict(max_num_residuals=BIG, frame_id=frame_id, threshold_translation_norm=thr_t)
    oprm, prm = O.r3live_params(**kw), capi.r3live_params(**kw)
    P = synth.prior_covariance()
    ref = om.update_iekf(sw.raw_xyz, O.Eskf(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=P.copy()), sw.t_last, oprm)
    est, trace, done = _run_product_host_loop(om, sw, oprm, prm, P)
    assert trace.shape[0] == ref["passes"]
    assert np.allclose(trace, ref["trace"], rtol=1e-9, atol=1e-12)
    for f in ("p", "q", "v", "ba", "bg", "g"):
        assert np.allclose(getattr(est, f), getattr(ref["eskf"], f), rtol=1e-10, atol=1e-12), f
    assert np.allclose(est.cov, ref["eskf"].cov, rtol=1e-8, atol=1e-12)
    assert done == (2 if thr_t > 0 else 1)


@pytest.mark.parametrize("kw", [dict(max_num_residuals=BIG), dict(max_num_residuals=BIG, threshold_translation_norm=0.0), dict(max_num_residuals=600)])
def test_iekf_host_algebra_matches_the_compiled_reference(ref_out, small_world, kw):
    """The product's host ESIKF algebra (srl_iekf_begin / srl_iekf_step in libsrlivo_b200.so, driven here by oracle passes so that
    it runs without a GPU) against lioOptimization::updateIEKF of the reference's own src/optimize.cpp (oracle/_ref/libsrl_reference.so)."""
    om, sw = small_world["omap"], small_world["sweep"]
    oprm, prm = O.r3live_params(**kw), capi.r3live_params(**kw)
    P = synth.prior_covariance()

    def rec():
        ref = Rf.Reference()
        ref.load(*om.snapshot())
        res = ref.update_iekf(sw.raw_xyz, O.Eskf(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=P.copy()), sw.t_last, oprm)
        return dict(success=res["success"], threw=res["threw"], frame_q=res["frame_q"], frame_t=res["frame_t"], **eskf_fields(res["eskf"]))
    r = ref_out("iekf." + "_".join(f"{k}{v}" for k, v in sorted(kw.items())), rec)
    est, trace, done = _run_product_host_loop(om, sw, oprm, prm, P)
    assert r["success"] and not r["threw"]
    for f in ("p", "q", "v", "ba", "bg", "g"):
        assert np.allclose(getattr(est, f), r[f], rtol=1e-9, atol=1e-11), f
    assert np.allclose(est.cov, r["cov"], rtol=1e-6, atol=1e-11)
    assert np.allclose(trace[-1][17:20], r["frame_t"], rtol=0, atol=1e-11) and np.allclose(trace[-1][20:24], r["frame_q"], rtol=0, atol=1e-11)


def test_host_plane_fit_matches_numpy():
    rng = np.random.default_rng(9)
    for trial in range(200):
        P = rng.normal(size=(20, 3)) * np.array([0.5, 0.4, 0.01 * (1 + trial % 5)])
        P = (P @ np.linalg.qr(rng.normal(size=(3, 3)))[0].T + rng.normal(size=3) * 30).astype(np.float32).astype(np.float64)
        n = np.zeros(3); a2d = C.c_double(0); ev = np.zeros(3)
        assert capi.lib().srl_host_plane_fit(capi.ptr(P), 20, capi.ptr(n), C.byref(a2d), capi.ptr(ev)) == 0
        Q = P - P.mean(0)
        w, V = np.linalg.eigh(Q.T @ Q)
        assert np.allclose(ev, w, rtol=1e-9, atol=1e-12 * w.max())
        assert abs(abs(n @ V[:, 0]) - 1) < 1e-9
        assert abs(a2d.value - (np.sqrt(w[1]) - np.sqrt(abs(w[0]))) / np.sqrt(w[2])) < 1e-9


def test_host_plane_fit_and_observe_match_the_compiled_reference(ref_out):
    """srl_host_plane_fit (the plane fit of srl_math.cuh compiled for the host) and srl_eskf_observe against the reference's own
    computeNeighborhoodDistribution (src/optimize.cpp:316-353) and eskfEstimator::observe (src/eskfEstimator.cpp:219-230)."""
    rng = np.random.default_rng(19)
    sets = []
    for trial in range(200):
        P = rng.normal(size=(20, 3)) * np.array([0.5, 0.4, 0.01 * (1 + trial % 5)])
        sets.append((P @ np.linalg.qr(rng.normal(size=(3, 3)))[0].T + rng.normal(size=3) * 30).astype(np.float32).astype(np.float64))

    def rec():
        ref = Rf.Reference()
        out = [ref.neighborhood(P) for P in sets]
        return dict(rc=np.array([rc for rc, _ in out]), normal=np.stack([nh["normal"] for _, nh in out]), a2D=np.array([nh["a2D"] for _, nh in out]))
    r = ref_out("neighborhood", rec)
    for trial, P in enumerate(sets):
        n = np.zeros(3); a2d = C.c_double(0); ev = np.zeros(3)
        assert capi.lib().srl_host_plane_fit(capi.ptr(P), 20, capi.ptr(n), C.byref(a2d), capi.ptr(ev)) == 0
        assert r["rc"][trial] == 0
        a2d_ref = r["a2D"][trial]
        assert abs(abs(n @ r["normal"][trial]) - 1) < 1e-9 and abs(a2d.value - a2d_ref) <= 1e-9 * max(1.0, abs(a2d_ref))
    cases = []
    for trial in range(30):
        scale = [0.05, 1e-6, 0.5][trial % 3]
        kw = dict(p=rng.normal(size=3), q=synth.quat_from_rotvec(rng.normal(size=3)), v=rng.normal(size=3), ba=rng.normal(size=3) * 0.01,
                  bg=rng.normal(size=3) * 0.01, g=np.array([0.3, -0.2, 9.7]) + rng.normal(size=3) * 0.1)
        cases.append((kw, rng.normal(size=17) * scale))
    names = ("p", "q", "v", "ba", "bg", "g")
    r = ref_out("observe", lambda: {f: np.stack([getattr(Rf.eskf_observe(O.Eskf(**kw), dx), f) for kw, dx in cases]) for f in names})
    for trial, (kw, dx) in enumerate(cases):
        a = lio.EskfEstimator(**kw).observe(dx)
        for f in names:
            assert np.allclose(getattr(a, f), r[f][trial], rtol=0, atol=1e-14), f


def test_shard_ranges_cover_the_sweep_in_order():
    for n in (0, 1, 31, 32, 33, 100000, 100001, 499999):
        for world in (1, 2, 3, 4, 8):
            prev = 0
            for r in range(world):
                b, e = dist.shard_range(n, r, world)
                assert b == prev and b <= e and (b % 32 == 0 or b == n)
                prev = e
            assert prev == n


_WORKER = r'''
import os, sys
sys.path.insert(0, sys.argv[1])
import numpy as np, torch, torch.distributed as dist_
import ctypes as C
from oracle import oracle_py as O
from sr_livo_b200 import capi, dist, lio, synth
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist_.init_process_group("gloo", rank=rank, world_size=world)
pts = synth.sample_map_points(80.0, 60.0, seed=1)
sw = synth.make_sweep(3000, seed=1000, yaw=0.5)
om = O.OracleMap(); om.add_points(pts)               # replicated map on every rank
kw = dict(max_num_residuals=2**31-1)
oprm, prm = O.r3live_params(**kw), capi.r3live_params(**kw)
b, e = dist.shard_range(sw.raw_xyz.shape[0], rank, world)
def pass_fn(fq, ft):                                  # this rank's shard, as the GPU pass would produce it
    r = om.build_plane_residuals(sw.raw_xyz[b:e], fq, ft, sw.t_last, oprm)
    blk = np.zeros(32)
    iu = np.triu_indices(6)
    blk[:21] = r.HTH[iu]; blk[21:27] = r.HTh; blk[27] = r.loss_sum; blk[28] = r.num_residuals
    blk[29] = r.num_full_neighborhoods; blk[30] = r.sum_candidates
    return torch.from_numpy(blk)
st = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=synth.prior_covariance()).to_c()
fq, ft = sw.q_init.copy(), sw.t_init.copy()
out = dist.iekf_loop(pass_fn, st, fq, ft, prm)
est = lio.EskfEstimator.from_c(st)
ref = om.update_iekf(sw.raw_xyz, O.Eskf(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=synth.prior_covariance()), sw.t_last, oprm)
assert out["passes"] == ref["passes"], (out["passes"], ref["passes"])
assert np.allclose(est.p, ref["eskf"].p, atol=1e-9) and np.allclose(est.q, ref["eskf"].q, atol=1e-9)
assert np.allclose(est.cov, ref["eskf"].cov, rtol=1e-6, atol=1e-12)
# every rank ends in the same state, bit for bit
t = torch.from_numpy(np.concatenate([est.p, est.q, est.cov.reshape(-1)]))
lst = [torch.zeros_like(t) for _ in range(world)]
dist_.all_gather(lst, t)
assert all(torch.equal(lst[0], x) for x in lst)
dist_.destroy_process_group()
print("rank", rank, "ok")
'''


def test_sharded_iekf_loop_world_size_2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    port = 29500 + (os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script), ROOT], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=300)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o


def test_cpp_adapter_header_compiles_and_fails_loudly_without_a_gpu(tmp_path):
    """include/srlivo_b200_lio.hpp (the C++ host mirror a maintainer includes) builds against the library with the
    reference's own language level (-std=c++14) and, on a box without a GPU, construction throws instead of falling
    back to anything."""
    import torch
    src = tmp_path / "adapter.cpp"
    src.write_text(r'''
#include <cstdio>
#include "srlivo_b200_lio.hpp"
int main() {
    try {
        srl::LioBackend lio(0, nullptr, 1 << 12, 1 << 12);
        srl_icp_params p; srl_icp_params_r3live(&p);
        std::printf("constructed mapSize=%lld K=%d\n", lio.mapSize(), p.max_number_neighbors);
        return 0;
    } catch (const std::exception& e) { std::printf("threw: %s\n", e.what()); return 3; }
}''')
    exe = tmp_path / "adapter"
    libdir = os.path.dirname(capi.LIB_PATH)
    subprocess.check_call(["g++", "-std=c++14", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L", libdir, "-lsrlivo_b200", f"-Wl,-rpath,{libdir}"])
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    if torch.cuda.is_available():
        assert r.returncode == 0 and "constructed mapSize=0 K=20" in r.stdout
    else:
        assert r.returncode == 3 and "no CPU fallback" in r.stdout


@pytest.mark.parametrize("arm", ["reference", "port"])
def test_bench_reference_arm_prints_the_contract_line(arm):
    """bench.py --impl reference runs on the CPU only (no GPU) and prints one JSON line with the contract's keys: the reference's
    own sources compiled where they lie (oracle/_ref/libsrl_reference.so) when that library exists, else / on request the oracle port."""
    import json
    from oracle import reference_py as Rf
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--points", "3000", "--map-extent", "80"], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, SRL_CPU_ARM=arm))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    with_ref = arm == "reference" and Rf.available()
    cb = line["cpu_baseline"]
    assert line["impl"] == "reference" and cb["cores"] >= 1
    if with_ref:   # both CPU forms are timed, the faster one is the value
        assert cb["kind"] in ("reference", "port") and cb["value"] == max(cb["reference_value"], cb["port_value"])
    else:
        assert cb["kind"] == "port"
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"] and line["value"] > 0
    assert "workload" in line["config"]
    if with_ref:
        assert cb["pose_equals_port"] is True


def test_c_shard_range_matches_the_python_one():
    """srl_shard_range (what srl_optimize_host_dist uses) == dist.shard_range (what the Python loop uses)."""
    import ctypes as C
    from sr_livo_b200 import dist
    L = capi.lib()
    for n in (0, 1, 31, 32, 33, 1000, 12345, 100000, 500000):
        for world in (1, 2, 3, 4, 8):
            for r in range(world):
                b, e = C.c_size_t(0), C.c_size_t(0)
                L.srl_shard_range(n, r, world, C.byref(b), C.byref(e))
                assert (b.value, e.value) == dist.shard_range(n, r, world)


def test_python_mirror_marshals_the_state_into_persistent_buffers():
    """LioOptimization._marshal / _unmarshal: the srl_eskf_state view and the pose block carry exactly what to_c() carried."""
    from sr_livo_b200 import lio

    class Bare(lio.LioOptimization):
        def __init__(self):
            self.R_imu_lidar = np.arange(9.0).reshape(3, 3)
            self.t_imu_lidar = np.array([0.1, 0.2, 0.3])
            self.eskf_pro = lio.EskfEstimator(p=np.array([1.0, 2.0, 3.0]), q=np.array([0.1, 0.2, 0.3, 0.9]), v=np.array([4.0, 5.0, 6.0]),
                                              ba=np.array([7.0, 8.0, 9.0]), bg=np.array([1.5, 2.5, 3.5]), g=np.array([0.0, 0.1, 9.8]),
                                              cov=np.arange(289.0).reshape(17, 17))
            self.ctx = None
    L = Bare()
    b = L._call_buffers()
    L._marshal(b, [9.0, 8.0, 7.0], None, [5.0, 5.5, 6.0])
    ref = L.eskf_pro.to_c()
    for f in ("p", "q", "v", "ba", "bg", "g", "cov"):
        assert list(getattr(b["st"], f)) == list(getattr(ref, f)), f
    blk = b["blk"]
    assert np.array_equal(blk[0:4], L.eskf_pro.q) and np.array_equal(blk[4:7], [5.0, 5.5, 6.0]) and np.array_equal(blk[7:10], [9.0, 8.0, 7.0])
    assert np.array_equal(blk[10:19], np.arange(9.0)) and np.array_equal(blk[19:22], [0.1, 0.2, 0.3])
    assert L._call_buffers() is b                                    # built once
