"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs.

Bar (BASELINE.json north_star): point-to-voxel association bit-exact (status + the 20 neighbour ids per keypoint,
in order); residuals / Jacobians / normal equations / state within 1e-5 relative.
"""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle_py as O
from sr_livo_b200 import synth

pytestmark = pytest.mark.gpu
BIG = 2 ** 31 - 1
REL = 1e-5
# the cases of the comparisons with the compiled reference (its outputs: tests/test_reference_pin.py, test_small_world_*)
SMALL_WORLD_PASS = [dict(max_num_residuals=BIG), dict(max_num_residuals=BIG, frame_id=5), dict(max_num_residuals=600)]
SMALL_WORLD_UPDATE = [dict(max_num_residuals=BIG), dict(max_num_residuals=600)]


@pytest.fixture(scope="module")
def L():
    from sr_livo_b200 import lio
    obj = lio.LioOptimization(max_voxels=1 << 18, sweep_capacity=1 << 17)
    yield obj
    obj.close()


def _map_dict(keys, counts, xyz):
    return {tuple(k): x[:c].copy() for k, c, x in zip(keys.tolist(), counts.tolist(), xyz)}


def _assert_map_equal(L, om):
    g = _map_dict(*L.voxel_map.download())
    o = _map_dict(*om.snapshot())
    assert g.keys() == o.keys()
    bad = [k for k in o if not np.array_equal(g[k], o[k])]
    assert not bad, bad[:5]
    assert L.voxel_map.stats() == (om.num_voxels, om.num_points)


def _assert_pass_equal(g, o, full_cov=True):
    assert o.num_fragile == 0
    assert np.array_equal(g.status, o.status)
    full = o.status >= 1
    assert np.array_equal(g.nbr[full], o.nbr[full])
    assert np.array_equal(g.world_xyz[o.status >= 0], o.world_xyz[o.status >= 0])   # same op order, no FMA: bit-exact
    assert np.array_equal(g.nbr_dist[full], o.nbr_dist[full])
    assert g.num_residuals == o.num_residuals and g.num_full_neighborhoods == o.num_full_neighborhoods
    if full.any():
        ref, got = o.plane[full], g.plane[full]
        scale = np.maximum(np.abs(ref).max(axis=0), 1e-12)
        assert np.all(np.abs(got - ref) <= REL * scale)
    if o.num_residuals:
        assert np.abs(g.HTH - o.HTH).max() <= REL * np.abs(o.HTH).max()
        assert np.abs(g.HTh - o.HTh).max() <= REL * max(np.abs(o.HTh).max(), 1e-12)
        assert abs(g.loss_sum - o.loss_sum) <= REL * o.loss_sum
    assert g.success == o.success


# ---- map: K3 insert / K4 mirror ---------------------------------------------------------------------------------
def test_map_insert_matches_oracle_including_second_sweep(L, small_world):
    L.voxel_map.clear()
    om = O.OracleMap()
    pts = small_world["pts"]
    assert L.addPointsToMap(pts) == om.add_points(pts)
    _assert_map_equal(L, om)
    for i in range(3):   # three registered sweeps into the populated map (present-voxel path, order dependence)
        sw = synth.make_sweep(15000, seed=1100 + i, yaw=0.3 * i, position=(1.0 * i, 3.0, 1.8))
        reg = synth.registered_points(sw)
        assert L.addPointsToMap(reg) == om.add_points(reg)
    _assert_map_equal(L, om)
    # offering the same points again adds nothing (distance 0 to themselves): idempotence
    assert L.addPointsToMap(reg) == 0 == om.add_points(reg)


def test_map_insert_edge_cases(L):
    L.voxel_map.clear()
    om = O.OracleMap()
    assert L.addPointsToMap(np.zeros((0, 3))) == 0                              # empty batch
    rng = np.random.default_rng(4)
    neg = rng.uniform(-3, 3, (5000, 3))                                         # keys -2..2 incl. the double-width cell 0
    assert L.addPointsToMap(neg, min_distance_points=0.05) == om.add_points(neg, min_distance_points=0.05)
    one = np.array([[100.25, -7.5, 3.125]])
    assert L.addPointsToMap(one) == om.add_points(one) == 1
    dup = np.repeat(one, 50, axis=0)                                            # same point 50 times in one batch
    assert L.addPointsToMap(dup) == om.add_points(dup) == 0
    edge = np.array([[0.99999999999, 0.1, 0.1], [-0.99999999999, 0.1, 0.1]])    # float rounding moves the key
    assert L.addPointsToMap(edge) == om.add_points(edge)
    far = rng.uniform(-3, 3, (300, 3)) + 500.0
    assert L.addPointsToMap(far, min_num_points=1) == om.add_points(far, min_num_points=1) == 0   # never creates voxels
    grow = rng.uniform(-3, 3, (3000, 3))
    assert L.addPointsToMap(grow, min_distance_points=0.05, min_num_points=3) == om.add_points(grow, min_distance_points=0.05, min_num_points=3)
    _assert_map_equal(L, om)


def test_map_upload_download_roundtrip(L, small_world):
    om = small_world["omap"]
    keys, counts, xyz = om.snapshot()
    L.voxel_map.upload(keys, counts, xyz)
    _assert_map_equal(L, om)
    from sr_livo_b200 import capi
    with pytest.raises(capi.SrlError):                                            # duplicate keys are rejected
        L.voxel_map.upload(np.concatenate([keys[:4], keys[:1]]), np.concatenate([counts[:4], counts[:1]]),
                           np.concatenate([xyz[:4], xyz[:1]]))


def test_map_full_is_reported():
    from sr_livo_b200 import capi, lio
    ctx = lio.Context(0)
    m = lio.VoxelHashMap(ctx, max_voxels=8)
    pts = np.stack([np.arange(20) + 0.5, np.full(20, 0.5), np.full(20, 0.5)], 1)
    with pytest.raises(capi.SrlError) as ei:
        m.insert(pts)
    assert ei.value.code == capi.SRL_MAP_FULL
    assert m.stats() == (0, 0)                                                    # nothing was mutated
    m.close(); ctx.close()


# ---- one pass ---------------------------------------------------------------------------------------------------
def _load_world(L, world):
    keys, counts, xyz = world["omap"].snapshot()
    L.voxel_map.upload(keys, counts, xyz)
    return world["omap"], world["sweep"]


@pytest.mark.parametrize("kw", [
    dict(max_num_residuals=BIG),                                   # steady state nb=1
    dict(max_num_residuals=BIG, frame_id=5),                       # init frames: nb=2, thr=1
    dict(max_num_residuals=600),                                   # r3live.yaml cap
    dict(max_num_residuals=-1),                                    # compiled default: stops after first full keypoint
    dict(max_num_residuals=BIG, threshold_voxel_occupancy=15),     # sparse voxels ignored
    dict(max_num_residuals=BIG, max_number_neighbors=10, min_number_neighbors=10),
    dict(max_num_residuals=BIG, max_number_neighbors=20, min_number_neighbors=5),
    dict(max_num_residuals=BIG, power_planarity=1.5, max_dist_to_plane_icp=0.05, weight_alpha=0.5, weight_neighborhood=0.5),
    dict(max_num_residuals=BIG, voxel_neighborhood=0),
])
def test_pass_matches_oracle(L, small_world, kw):
    from sr_livo_b200 import lio
    om, sw = _load_world(L, small_world)
    L.setKeypoints(sw.raw_xyz)
    g = L.buildPlaneResiduals(lio.r3live_params(**kw), sw.q_init, sw.t_init, sw.t_last, debug=True)
    o = om.build_plane_residuals(sw.raw_xyz, sw.q_init, sw.t_init, sw.t_last, O.r3live_params(**kw), debug=True)
    _assert_pass_equal(g, o)


def test_single_launch_sweep_order_is_the_cub_order(L, small_world):
    """The thread-block-cluster radix sort (k_sweep_order_cluster) orders a sweep exactly like the CUB sort it replaces: the
    library runs both for the first uses after the option is set and keeps the cluster kernel only if the orders are
    identical on the device (counter 1; 0 = it fell back to CUB).  Sizes: a full cluster (131072), the bench sweep, a
    handful of points, a ragged size; 150000 exceeds what 16 CTAs hold in registers and goes through CUB without
    retiring the kernel.  The pass sums are summed in sweep order, so they are bit-identical under either sort."""
    from sr_livo_b200 import lio
    L = lio.LioOptimization(max_voxels=1 << 18, sweep_capacity=160000)   # the shared fixture stops at 131072 points
    om, sw = _load_world(L, small_world)
    rng = np.random.default_rng(11)
    prm = lio.r3live_params(max_num_residuals=BIG)
    try:
        L.ctx.set_option("cluster_order", 1)
        for n in (131072, 100000, 7, 40001, 150000, 1000):
            raw = rng.uniform(-140.0, 140.0, size=(n, 3))          # beyond +-128 m: clamped cells
            raw[: n // 2] = sw.raw_xyz[rng.integers(0, sw.raw_xyz.shape[0], n // 2)]
            L.setKeypoints(raw)
            L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last)
        assert L.ctx.counter("cluster_order_active") == 1
        out = {}
        for mode in (1, 0):
            L.ctx.set_option("cluster_order", mode)
            L.setKeypoints(sw.raw_xyz)
            out[mode] = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last)
        assert np.array_equal(out[1].HTH, out[0].HTH) and np.array_equal(out[1].HTh, out[0].HTh)
        assert out[1].num_residuals == out[0].num_residuals
    finally:
        L.ctx.set_option("cluster_order", 1)


def _close(a, b, rel=1e-12):
    return np.abs(a - b).max() <= rel * np.abs(b).max()


@pytest.mark.parametrize("kw", [dict(max_num_residuals=BIG), dict(max_num_residuals=BIG, frame_id=5)])
def test_exact_selection_path_matches_oracle(L, small_world, kw):
    """Three ways to the same answer: (a) auto = k1_scan + k1_fit (FP32 packed keys + guards + exact finish) where
    applicable, (b) k1_assoc only (FP32 selection with error bound, exact fallback), (c) k1_assoc with the exact FP64 selection
    forced for every keypoint.  All must equal the oracle: ids bit-exact, floats to rounding."""
    from sr_livo_b200 import lio
    om, sw = _load_world(L, small_world)
    n = 1500
    L.setKeypoints(sw.raw_xyz[:n])
    o = om.build_plane_residuals(sw.raw_xyz[:n], sw.q_init, sw.t_init, sw.t_last, O.r3live_params(**kw), debug=True)
    prm = lio.r3live_params(**kw)
    g_auto = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last, debug=True)
    L.ctx.set_option("k1_variant", 2)
    try:
        before = L.ctx.counter("exact_fallbacks")
        g_v2 = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last, debug=True)
        mid = L.ctx.counter("exact_fallbacks")
        L.ctx.set_option("force_exact_selection", 1)
        g_exact = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last, debug=True)
        after = L.ctx.counter("exact_fallbacks")
    finally:
        L.ctx.set_option("force_exact_selection", 0)
        L.ctx.set_option("k1_variant", 0)
    for g in (g_auto, g_v2, g_exact):
        _assert_pass_equal(g, o)
    assert np.array_equal(g_auto.nbr, g_exact.nbr) and np.array_equal(g_v2.nbr, g_exact.nbr)
    assert _close(g_auto.HTH, g_exact.HTH) and _close(g_v2.HTH, g_exact.HTH)
    n_cand = int((o.num_candidates >= 20).sum())
    assert after - mid == n_cand                       # forced: every keypoint with >= K candidates went the exact way
    assert mid - before <= 0.1 * n_cand                # normal: the FP32 selection decides almost all of them


def test_fast_kernel_hands_ambiguous_keypoints_to_the_exact_kernel(L, small_world):
    """k1_fast flags what it cannot certify; k1_assoc redoes those and adds k1_fast's sums.  With the guard entries the
    natural rate is ~0, so the hand-over is also forced on every 7th keypoint."""
    from sr_livo_b200 import lio
    om, sw = _load_world(L, small_world)
    prm = lio.r3live_params(max_num_residuals=BIG)
    L.setKeypoints(sw.raw_xyz)
    o = om.build_plane_residuals(sw.raw_xyz, sw.q_init, sw.t_init, sw.t_last, O.r3live_params(max_num_residuals=BIG), debug=True)
    a0 = L.ctx.counter("fast_ambiguous")
    g = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last, debug=True)
    a1 = L.ctx.counter("fast_ambiguous")
    _assert_pass_equal(g, o)
    assert a1 - a0 <= 0.002 * sw.raw_xyz.shape[0]
    L.ctx.set_option("fast_force_ambiguous_mod", 7)
    try:
        g7 = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last, debug=True)
        a2 = L.ctx.counter("fast_ambiguous")
    finally:
        L.ctx.set_option("fast_force_ambiguous_mod", 0)
    _assert_pass_equal(g7, o)
    assert a2 - a1 >= int((o.num_candidates[::7] >= 20).sum())
    assert _close(g7.HTH, g.HTH) and g7.num_residuals == g.num_residuals


@pytest.mark.parametrize("split_lpk", [4, 2])
def test_split_scan_fit_form_matches_oracle(L, small_world, cfg1_world, split_lpk):
    """k1_scan (2 or 4 lanes per keypoint, short per-lane lists, merge) + k1_fit: same neighbour lists, same sums, and
    the same hand-over of uncertified keypoints to the exact kernel."""
    from sr_livo_b200 import lio
    prm, oprm = lio.r3live_params(max_num_residuals=BIG), O.r3live_params(max_num_residuals=BIG)
    L.ctx.set_option("k1_variant", 3)
    L.ctx.set_option("split_lanes_per_keypoint", split_lpk)
    try:
        for world, n in ((small_world, None), (cfg1_world, 20000)):
            om, sw = _load_world(L, world)
            raw = sw.raw_xyz if n is None else sw.raw_xyz[:n]
            L.setKeypoints(raw)
            o = om.build_plane_residuals(raw, sw.q_init, sw.t_init, sw.t_last, oprm, nthreads=8, debug=True)
            a0 = L.ctx.counter("fast_ambiguous")
            g = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last, debug=True)
            a1 = L.ctx.counter("fast_ambiguous")
            _assert_pass_equal(g, o)
            assert a1 - a0 <= 0.01 * raw.shape[0]
            g2 = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last)
            g3 = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last)
            assert g2.num_residuals == o.num_residuals and _close(g2.HTH, o.HTH) and _close(g2.HTh, o.HTh)
            assert np.array_equal(g2.HTH, g3.HTH) and np.array_equal(g2.HTh, g3.HTh)     # run-to-run deterministic
            assert 0 < g2.num_candidates_scanned <= o.sum_candidates
            L.ctx.set_option("fast_force_ambiguous_mod", 5)
            try:
                g5 = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last, debug=True)
            finally:
                L.ctx.set_option("fast_force_ambiguous_mod", 0)
            _assert_pass_equal(g5, o)
            assert L.ctx.counter("fast_ambiguous") - a1 >= int((o.num_candidates[::5] >= 20).sum())
        # ragged tail / tiny sweeps
        om, sw = _load_world(L, small_world)
        for n in (1, 7, 33, 1001):
            L.setKeypoints(sw.raw_xyz[:n])
            o = om.build_plane_residuals(sw.raw_xyz[:n], sw.q_init, sw.t_init, sw.t_last, oprm, debug=True)
            _assert_pass_equal(L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last, debug=True), o)
    finally:
        L.ctx.set_option("k1_variant", 0)
        L.ctx.set_option("split_lanes_per_keypoint", 4)


@pytest.mark.parametrize("lpk", [1, 2, 4])
def test_fast_kernel_lanes_per_keypoint_variants(L, small_world, lpk):
    """k1_fast deals a keypoint's candidates to 1, 2 or 4 lanes and merges their top lists: same answer every way."""
    from sr_livo_b200 import lio
    om, sw = _load_world(L, small_world)
    prm = lio.r3live_params(max_num_residuals=BIG)
    L.setKeypoints(sw.raw_xyz[:3001])
    o = om.build_plane_residuals(sw.raw_xyz[:3001], sw.q_init, sw.t_init, sw.t_last, O.r3live_params(max_num_residuals=BIG), debug=True)
    L.ctx.set_option("k1_variant", 1)                 # k1_fast, the thread-per-keypoint form (not the default any more)
    L.ctx.set_option("fast_lanes_per_keypoint", lpk)
    try:
        a0 = L.ctx.counter("fast_ambiguous")
        g = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last, debug=True)
        g2 = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last)
        L.ctx.set_option("fast_force_ambiguous_mod", 9)          # and its hand-over to the exact kernel
        g9 = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last, debug=True)
        a1 = L.ctx.counter("fast_ambiguous")
    finally:
        L.ctx.set_option("fast_force_ambiguous_mod", 0)
        L.ctx.set_option("fast_lanes_per_keypoint", 1)
        L.ctx.set_option("k1_variant", 0)
    _assert_pass_equal(g, o)
    _assert_pass_equal(g9, o)
    assert a1 - a0 >= int((o.num_candidates[::9] >= 20).sum())
    assert g2.num_residuals == o.num_residuals and _close(g2.HTH, o.HTH)


@pytest.mark.parametrize("size,cap_pts", [(0.5, 20), (2.0, 20), (0.7, 12)])
def test_other_voxel_sizes_and_caps(size, cap_pts):
    """Nothing in the kernels may assume the 1 m / 20-point configuration the reference ships: map insert, keys, cell
    lower bounds and the FP32 error window all scale with size_voxel_map (0.7 is not exactly representable)."""
    from sr_livo_b200 import lio
    pts = synth.sample_map_points(80.0, 120.0 if size < 1 else 40.0, seed=5)
    sw = synth.make_sweep(3000, seed=1005, yaw=0.4)
    Lx = lio.LioOptimization(max_voxels=1 << 19, sweep_capacity=4096, size_voxel_map=size, max_num_points_in_voxel=cap_pts)
    try:
        om = O.OracleMap()
        md = 0.15 * size
        assert Lx.addPointsToMap(pts, min_distance_points=md) == om.add_points(pts, voxel_size=size, max_num_points_in_voxel=cap_pts,
                                                                               min_distance_points=md)
        g_keys, g_cnt, g_xyz = Lx.voxel_map.download()
        o_keys, o_cnt, o_xyz = om.snapshot(cap=cap_pts)
        gd, od = _map_dict(g_keys, g_cnt, g_xyz), _map_dict(o_keys, o_cnt, o_xyz)
        assert gd.keys() == od.keys() and all(np.array_equal(gd[k], od[k]) for k in od)
        kw = dict(max_num_residuals=BIG, size_voxel_map=size, max_dist_to_plane_icp=0.3 * size)
        Lx.setKeypoints(sw.raw_xyz)
        for extra in (dict(), dict(frame_id=5)):
            g = Lx.buildPlaneResiduals(lio.r3live_params(**kw, **extra), sw.q_init, sw.t_init, sw.t_last, debug=True)
            o = om.build_plane_residuals(sw.raw_xyz, sw.q_init, sw.t_init, sw.t_last, O.r3live_params(**kw, **extra), debug=True)
            _assert_pass_equal(g, o)
            assert o.num_full_neighborhoods > 300
    finally:
        Lx.close()


def test_pass_config1_20k_points_200k_map(L, cfg1_world):
    """BASELINE config 1: 20k-pt sweep, ~200k-pt map, 1 ESIKF iteration, r3live params (cap lifted and cap 600)."""
    from sr_livo_b200 import lio
    om, sw = _load_world(L, cfg1_world)
    assert 150_000 < om.num_points < 260_000
    L.setKeypoints(sw.raw_xyz)
    for cap in (BIG, 600):
        g = L.buildPlaneResiduals(lio.r3live_params(max_num_residuals=cap), sw.q_init, sw.t_init, sw.t_last, debug=True)
        o = om.build_plane_residuals(sw.raw_xyz, sw.q_init, sw.t_init, sw.t_last, O.r3live_params(max_num_residuals=cap), debug=True)
        _assert_pass_equal(g, o)


def test_pass_extrinsics_and_unnormalised_quaternion(L, small_world):
    """R_il / t_il are applied before the pose; the distance/Jacobian use the UN-normalised quaternion (src/optimize.cpp:95)."""
    from sr_livo_b200 import lio
    om, sw = _load_world(L, small_world)
    R_il = synth.quat_to_rot(synth.quat_from_rotvec([0.02, -0.01, 0.03]))
    t_il = np.array([0.05, -0.02, 0.1])
    raw = (sw.raw_xyz - t_il) @ R_il            # so that R_il raw + t_il == the original body points
    q = sw.q_init * 1.0000003                    # slightly un-normalised, as after many compositions
    L.R_imu_lidar, L.t_imu_lidar = R_il, t_il
    try:
        L.setKeypoints(raw)
        g = L.buildPlaneResiduals(lio.r3live_params(max_num_residuals=BIG), q, sw.t_init, sw.t_last, debug=True)
    finally:
        L.R_imu_lidar, L.t_imu_lidar = np.eye(3), np.zeros(3)
    o = om.build_plane_residuals(raw, q, sw.t_init, sw.t_last, O.r3live_params(max_num_residuals=BIG), R_il=R_il, t_il=t_il, debug=True)
    _assert_pass_equal(g, o)


@pytest.mark.parametrize("n", [0, 1, 31, 32, 33, 257])
def test_pass_ragged_sizes(L, small_world, n):
    from sr_livo_b200 import lio
    om, sw = _load_world(L, small_world)
    raw = sw.raw_xyz[:n]
    if n == 0:
        L.sweep.upload(np.zeros((0, 3)))
        L.sweep.n = 0
        g = L.buildPlaneResiduals(lio.r3live_params(max_num_residuals=BIG), sw.q_init, sw.t_init, sw.t_last)
        assert g.num_residuals == 0 and not g.success and np.all(g.HTH == 0)
        return
    L.setKeypoints(raw)
    g = L.buildPlaneResiduals(lio.r3live_params(max_num_residuals=BIG), sw.q_init, sw.t_init, sw.t_last, debug=True)
    o = om.build_plane_residuals(raw, sw.q_init, sw.t_init, sw.t_last, O.r3live_params(max_num_residuals=BIG), debug=True)
    _assert_pass_equal(g, o)


def test_pass_keypoints_outside_the_map_and_empty_map(L, small_world):
    from sr_livo_b200 import lio
    om, sw = _load_world(L, small_world)
    raw = sw.raw_xyz[:500].copy()
    raw[::2] += 5000.0                                   # half of them nowhere near the map
    L.setKeypoints(raw)
    g = L.buildPlaneResiduals(lio.r3live_params(max_num_residuals=BIG), sw.q_init, sw.t_init, sw.t_last, debug=True)
    o = om.build_plane_residuals(raw, sw.q_init, sw.t_init, sw.t_last, O.r3live_params(max_num_residuals=BIG), debug=True)
    _assert_pass_equal(g, o)
    assert np.all(g.status[::2] == 0)
    L.voxel_map.clear()
    g = L.buildPlaneResiduals(lio.r3live_params(max_num_residuals=BIG), sw.q_init, sw.t_init, sw.t_last)
    assert g.num_residuals == 0 and not g.success       # SRL_TOO_FEW_RESIDUALS <-> summary.success = false


def test_pass_is_deterministic_and_shards_sum_to_the_whole(L, small_world):
    from sr_livo_b200 import dist, lio
    om, sw = _load_world(L, small_world)
    prm = lio.r3live_params(max_num_residuals=BIG)
    L.setKeypoints(sw.raw_xyz)
    a = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last)
    b = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last)
    assert np.array_equal(a.HTH, b.HTH) and np.array_equal(a.HTh, b.HTh) and a.loss_sum == b.loss_sum   # bitwise, run to run
    n = sw.raw_xyz.shape[0]
    for world in (2, 4, 8):
        HTH = np.zeros((6, 6)); HTh = np.zeros(6); res = 0
        for r in range(world):
            bgn, end = dist.shard_range(n, r, world)
            L.sweep.set_shard(bgn, end)
            p = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last)
            HTH += p.HTH; HTh += p.HTh; res += p.num_residuals
        L.sweep.set_shard(0, n)
        assert res == a.num_residuals
        assert np.abs(HTH - a.HTH).max() <= 1e-12 * np.abs(a.HTH).max()
        assert np.abs(HTh - a.HTh).max() <= 1e-11 * np.abs(a.HTh).max()


def test_async_pass_into_a_caller_buffer(L, small_world):
    import torch
    from sr_livo_b200 import capi, dist, lio
    om, sw = _load_world(L, small_world)
    prm = lio.r3live_params(max_num_residuals=BIG)
    L.setKeypoints(sw.raw_xyz)
    ref = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last)
    blk = torch.full((32,), -1.0, dtype=torch.float64, device="cuda:0")
    fr = lio.make_frame(sw.q_init, sw.t_init, sw.t_last)
    rc = capi.lib().srl_build_plane_residuals_async(L.ctx.h, L.voxel_map.h, L.sweep.h, C.byref(fr), C.byref(prm),
                                                    C.c_void_p(blk.data_ptr()))
    assert rc == 0
    L.ctx.synchronize()
    ne = dist.unpack_block(blk.cpu().numpy())
    assert np.array_equal(np.array(ne.HTH).reshape(6, 6), ref.HTH) and ne.num_residuals == ref.num_residuals
    # the cap is not available on the async form
    rc = capi.lib().srl_build_plane_residuals_async(L.ctx.h, L.voxel_map.h, L.sweep.h, C.byref(fr),
                                                    C.byref(lio.r3live_params()), C.c_void_p(blk.data_ptr()))
    assert rc == capi.SRL_BAD_ARG


def test_bad_arguments_are_rejected(L, small_world):
    from sr_livo_b200 import capi, lio
    om, sw = _load_world(L, small_world)
    L.setKeypoints(sw.raw_xyz[:64])
    for kw in (dict(max_number_neighbors=33), dict(max_number_neighbors=0), dict(min_number_neighbors=0),
               dict(voxel_neighborhood=3), dict(size_voxel_map=0.5)):
        with pytest.raises(capi.SrlError) as ei:
            L.buildPlaneResiduals(lio.r3live_params(**kw), sw.q_init, sw.t_init, sw.t_last)
        assert ei.value.code == capi.SRL_BAD_ARG


# ---- the iterated update ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kw", [dict(max_num_residuals=BIG), dict(max_num_residuals=600),
                                dict(max_num_residuals=BIG, frame_id=5, num_iters_icp=3),
                                dict(max_num_residuals=BIG, threshold_translation_norm=0.0)])
def test_update_iekf_matches_oracle(L, small_world, kw):
    from sr_livo_b200 import lio
    om, sw = _load_world(L, small_world)
    n = 1500 if kw.get("frame_id") == 5 else sw.raw_xyz.shape[0]
    raw = sw.raw_xyz[:n]
    P = synth.prior_covariance()
    L.setKeypoints(raw)
    L.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), v=np.array([0.3, 0.0, 0.0]), cov=P.copy())
    summ, fq, ft = L.updateIEKF(lio.r3live_params(**kw), sw.t_last)
    ref = om.update_iekf(raw, O.Eskf(p=sw.t_init.copy(), q=sw.q_init.copy(), v=np.array([0.3, 0.0, 0.0]), cov=P.copy()), sw.t_last,
                         O.r3live_params(**kw))
    assert summ.success == ref["success"] and summ.passes_run == ref["passes"]
    assert summ.num_residuals_used == ref["num_residuals_used"]
    assert np.allclose(summ.trace, ref["trace"], rtol=REL, atol=1e-9)
    e, r = L.eskf_pro, ref["eskf"]
    for f in ("p", "q", "v", "ba", "bg", "g"):
        assert np.allclose(getattr(e, f), getattr(r, f), rtol=REL, atol=1e-9), f
    assert np.allclose(e.cov, r.cov, rtol=1e-4, atol=1e-12)
    assert np.allclose(fq, ref["frame_q"], atol=1e-9) and np.allclose(ft, ref["frame_t"], atol=1e-9)
    if kw.get("max_num_residuals") == BIG and "frame_id" not in kw:
        assert np.linalg.norm(e.p - sw.t_true) < 0.01           # it actually registers the sweep


@pytest.mark.parametrize("kw", [dict(), dict(frame_id=5, num_iters_icp=3), dict(threshold_translation_norm=0.0),
                                dict(threshold_translation_norm=0.0, num_iters_icp=2), dict(num_iters_icp=0)])
def test_device_resident_loop_equals_host_driven_loop(L, small_world, kw):
    """Row N1: the persistent ESIKF block on the device (all passes enqueued at once, one host wait) against the round-1 host loop
    (srl_iekf_step per pass): same passes, same early exit, state to 1e-9 — the two differ only in how the gain is formed
    (one 6x6 inverse via the Woodbury identity instead of two 17x17 inverses)."""
    from sr_livo_b200 import lio
    om, sw = _load_world(L, small_world)
    n = 1500 if kw.get("frame_id") == 5 else sw.raw_xyz.shape[0]
    raw = sw.raw_xyz[:n]
    P = synth.prior_covariance()
    prm = lio.r3live_params(max_num_residuals=BIG, **kw)
    out = {}
    try:
        for mode in (1, 0):
            L.ctx.set_option("device_loop", mode)
            L.setKeypoints(raw)
            L.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), v=np.array([0.3, 0.0, 0.0]),
                                           ba=np.array([0.01, -0.02, 0.0]), cov=P.copy())
            launches0 = L.ctx.kernel_launches
            summ, fq, ft = L.updateIEKF(prm, sw.t_last)
            out[mode] = (summ, fq, ft, L.eskf_pro, L.ctx.kernel_launches - launches0)
    finally:
        L.ctx.set_option("device_loop", 1)
    (sd, qd, td, ed, _), (sh, qh, th, eh, _) = out[1], out[0]
    assert (sd.success, sd.passes_run, sd.converged, sd.num_residuals_used) == (sh.success, sh.passes_run, sh.converged, sh.num_residuals_used)
    assert np.allclose(sd.trace, sh.trace, rtol=1e-7, atol=1e-11)
    for f in ("p", "q", "v", "ba", "bg", "g"):
        assert np.allclose(getattr(ed, f), getattr(eh, f), rtol=1e-9, atol=1e-11), f
    assert np.allclose(ed.cov, eh.cov, rtol=1e-6, atol=1e-13)
    assert np.allclose(qd, qh, atol=1e-11) and np.allclose(td, th, atol=1e-11)


def test_update_iekf_reports_too_few_residuals(L, small_world):
    from sr_livo_b200 import lio
    om, sw = _load_world(L, small_world)
    L.setKeypoints(sw.raw_xyz[:5])
    L.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=synth.prior_covariance())
    summ, _, _ = L.updateIEKF(lio.r3live_params(max_num_residuals=BIG), sw.t_last)
    assert not summ.success and summ.passes_run == 1
    assert np.array_equal(L.eskf_pro.p, sw.t_init)            # state untouched, like the early return at src/optimize.cpp:155


def test_optimize_host_end_to_end(L, small_world):
    """optimize() with host buffers: H2D, updateIEKF, final re-transform of the frame (src/optimize.cpp:441-445)."""
    from sr_livo_b200 import lio
    om, sw = _load_world(L, small_world)
    L.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=synth.prior_covariance())
    summ, fq, ft, world = L.optimize(sw.raw_xyz, lio.r3live_params(max_num_residuals=BIG), sw.t_last)
    ref = om.update_iekf(sw.raw_xyz, O.Eskf(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=synth.prior_covariance()), sw.t_last,
                         O.r3live_params(max_num_residuals=BIG))
    assert summ.passes_run == ref["passes"] and np.allclose(ft, ref["frame_t"], atol=1e-9)
    expect = sw.raw_xyz @ O.quat_to_rot(fq).T + ft
    assert np.allclose(world, expect, rtol=0, atol=1e-10)
    # registered points go straight into the map, like stateEstimation (src/lioOptimization.cpp:1027)
    before = L.mapSize()
    added = L.addPointsToMap(world)
    assert L.mapSize() == before + added


def test_streaming_sweeps_insert_then_query(L, small_world):
    """BASELINE config 4: a stream of sweeps, each registered against the map (updateIEKF) and then inserted into it
    (stateEstimation, src/lioOptimization.cpp:992-1035); the sensor moves 1 m per sweep.  Poses after every sweep and the
    final map must equal the oracle doing the same thing point by point."""
    from sr_livo_b200 import lio
    pts = small_world["pts"]
    L.voxel_map.clear()
    om = O.OracleMap()
    assert L.addPointsToMap(pts) == om.add_points(pts)
    kw = dict(max_num_residuals=BIG)
    prm, oprm = lio.r3live_params(**kw), O.r3live_params(**kw)
    P = synth.prior_covariance()
    for i in range(5):
        sw = synth.make_sweep(6000, seed=1300 + i, yaw=0.5, position=(-6.0 + 1.0 * i, 3.0, 1.8))
        L.setKeypoints(sw.raw_xyz)
        L.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=P.copy())
        summ, fq, ft = L.updateIEKF(prm, sw.t_last)
        ref = om.update_iekf(sw.raw_xyz, O.Eskf(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=P.copy()), sw.t_last, oprm)
        assert summ.success and summ.passes_run == ref["passes"]
        assert np.allclose(ft, ref["frame_t"], atol=1e-9) and np.allclose(fq, ref["frame_q"], atol=1e-9)
        # the oracle inserts the points registered with ITS pose; the GPU inserts with the GPU pose: identical to ~1e-15,
        # so quantise the comparison through the oracle's own pose to keep the map check byte-exact
        fq, ft = ref["frame_q"].copy(), ref["frame_t"].copy()
        added = L.addSweepToMap(fq, ft)
        world = sw.raw_xyz @ O.quat_to_rot(fq).T + ft
        # same operation order as transformPoint: R*(R_il*raw + t_il) + t with the a0+(a1+a2) reductions
        R = O.quat_to_rot(fq)
        w = np.empty_like(sw.raw_xyz)
        for a in range(3):
            w[:, a] = (R[a, 0] * sw.raw_xyz[:, 0] + (R[a, 1] * sw.raw_xyz[:, 1] + R[a, 2] * sw.raw_xyz[:, 2])) + ft[a]
        assert np.allclose(w, world, atol=1e-12)
        assert added == om.add_points(w)
    _assert_map_equal(L, om)


def test_grid_sampling_matches_the_reference_order(L, small_world):
    """Row N2: gridSampling (src/utility.cpp:188-201).  Same keypoints in the same order as the reference's
    std::tr1::unordered_map walk (order matters: the max_num_residuals cap takes keypoints in that order)."""
    from sr_livo_b200 import lio
    sw = synth.make_sweep(60000, seed=1400, yaw=0.3)
    w = synth.registered_points(sw)
    for size in (1.5, 0.25, 7.0):
        g = L.gridSampling(w, size)
        o = O.grid_sampling(w, size)
        assert np.array_equal(g.astype(np.int64), o.astype(np.int64))
    assert L.gridSampling(np.zeros((0, 3)), 1.5).size == 0
    assert np.array_equal(L.gridSampling(w[:1], 1.5), [0])
    neg = -w[:5000]
    assert np.array_equal(L.gridSampling(neg, 1.5).astype(np.int64), O.grid_sampling(neg, 1.5).astype(np.int64))
    # end to end like optimize(): keypoints from gridSampling, then the capped update (r3live.yaml: 600 residuals)
    om, sw0 = _load_world(L, small_world)
    w0 = synth.registered_points(sw0, sw0.q_init, sw0.t_init)
    kp = L.gridSampling(w0, 0.4)
    assert np.array_equal(kp.astype(np.int64), O.grid_sampling(w0, 0.4).astype(np.int64)) and kp.size > 700
    raw = sw0.raw_xyz[kp]
    L.setKeypoints(raw)
    L.eskf_pro = lio.EskfEstimator(p=sw0.t_init.copy(), q=sw0.q_init.copy(), cov=synth.prior_covariance())
    summ, fq, ft = L.updateIEKF(lio.r3live_params(), sw0.t_last)
    ref = om.update_iekf(raw, O.Eskf(p=sw0.t_init.copy(), q=sw0.q_init.copy(), cov=synth.prior_covariance()), sw0.t_last, O.r3live_params())
    assert summ.passes_run == ref["passes"] and summ.num_residuals_used == ref["num_residuals_used"] == 600
    assert np.allclose(ft, ref["frame_t"], atol=1e-9) and np.allclose(fq, ref["frame_q"], atol=1e-9)
    # the frame may already live in HBM (device pointer): same sequence, no upload of the frame
    import ctypes as C
    import torch
    from sr_livo_b200 import capi
    world = sw0.raw_xyz @ O.quat_to_rot(sw0.q_init).T + sw0.t_init
    d_world = torch.from_numpy(np.ascontiguousarray(world)).cuda()
    out = np.zeros(world.shape[0], np.uint32)
    m = C.c_size_t(0)
    assert capi.lib().srl_grid_sampling(L.ctx.h, C.c_void_p(d_world.data_ptr()), world.shape[0], 0.5, capi.ptr(out), C.byref(m)) == 0
    assert np.array_equal(out[:m.value], L.gridSampling(world, 0.5))


def test_remove_points_far_from_location_then_keep_working(L, small_world):
    """Row N4 (src/lioOptimization.cpp:556-572): eviction by the voxel's first point, pool compaction and slot rebuild;
    the map must answer queries and take insertions afterwards exactly like the oracle's."""
    from sr_livo_b200 import lio
    keys, counts, xyz = small_world["omap"].snapshot()
    om = O.OracleMap(); om.load(keys, counts, xyz)            # a private copy: this test edits the map
    L.voxel_map.upload(keys, counts, xyz)
    sw = small_world["sweep"]
    loc = np.array([4.0, -3.0, 1.5])
    nv0, np0 = L.voxel_map.stats()
    assert L.removePointsFarFromLocation(loc, 1e4) == 0 and L.voxel_map.stats() == (nv0, np0)     # nothing is that far
    n_g = L.removePointsFarFromLocation(loc, 25.0)
    n_o = om.remove_far(loc, 25.0)
    assert n_g == n_o and 0 < n_g < nv0
    _assert_map_equal(L, om)
    assert L.mapSize() == om.num_points
    # queries against the shrunken map
    prm, oprm = lio.r3live_params(max_num_residuals=BIG), O.r3live_params(max_num_residuals=BIG)
    L.setKeypoints(sw.raw_xyz)
    _assert_pass_equal(L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last, debug=True),
                       om.build_plane_residuals(sw.raw_xyz, sw.q_init, sw.t_init, sw.t_last, oprm, debug=True))
    # and insertions: points land in evicted cells again
    reg = synth.registered_points(sw)
    assert L.addPointsToMap(reg) == om.add_points(reg)
    _assert_map_equal(L, om)
    # evict everything
    assert L.removePointsFarFromLocation(np.array([1e5, 0.0, 0.0]), 1.0) == om.remove_far(np.array([1e5, 0.0, 0.0]), 1.0)
    assert L.voxel_map.stats() == (0, 0) and om.num_voxels == 0
    L.voxel_map.clear()


def test_undistortion_and_sweep_end_transform_match_the_oracle(L):
    """Row N3 (src/utility.cpp:203-332): distortFrameByConstant, distortFrameByImu (incl. its one-iterator walk) and
    transformAllImuPoint, host buffers and device buffers, against the oracle."""
    import torch
    import ctypes as C
    from sr_livo_b200 import capi
    st = synth.make_imu_states()
    rng = np.random.default_rng(21)
    n = 50000
    raw = rng.normal(0, 30, (n, 3)); rel = synth.make_sweep_times(n)
    t0 = st[0]["timestamp"]
    R_il, t_il = L.R_imu_lidar, L.t_imu_lidar
    tol = dict(rtol=1e-12, atol=1e-10)                       # floating point: north_star allows 1e-5; libm differs in the last ulp

    o_c = O.distort_frame_by_constant(raw, rel, st, t0, R_il, t_il)
    g_c = L.distortFrameByConstant(raw, rel, st, t0)
    assert np.allclose(g_c, o_c, **tol) and np.abs(g_c - o_c).max() < 1e-11

    o_i, m_o = O.distort_frame_by_imu(raw, rel, st, t0, R_il, t_il)
    g_i, m_g = L.distortFrameByImu(raw, rel, st, t0)
    assert m_g == m_o == n and np.allclose(g_i, o_i, **tol)

    # the walk stops at the first point that fits no remaining interval; the rest keep the caller's values
    keep = np.full_like(raw, -3.0)
    for bad_at, val in ((1234, -1.0), (30000, 10.0), (40000, 1e6), (0, -50.0)):
        rel2 = rel.copy(); rel2[bad_at] = val
        o2, mo = O.distort_frame_by_imu(raw, rel2, st, t0, R_il, t_il, imu_xyz_in=keep)
        g2, mg = L.distortFrameByImu(raw, rel2, st, t0, imu_xyz_in=keep)
        assert mg == mo == bad_at and np.allclose(g2, o2, **tol) and np.all(g2[bad_at:] == -3.0)
    # unsorted but recoverable: a point one interval back after the walk moved on is NOT recoverable, one on the shared
    # boundary (within 1e-6 s of an IMU stamp) is
    ts = np.array([s_["timestamp"] for s_ in st])
    rel3 = rel.copy(); k = n // 2
    rel3[k] = (ts[np.searchsorted(ts, t0 + rel[k] / 1000.0) - 1] - t0) * 1000.0 + 5e-4      # just inside the lower boundary's tolerance
    o3, mo3 = O.distort_frame_by_imu(raw, rel3, st, t0, R_il, t_il, imu_xyz_in=keep)
    g3, mg3 = L.distortFrameByImu(raw, rel3, st, t0, imu_xyz_in=keep)
    assert mg3 == mo3 and np.allclose(g3, o3, **tol)

    o_t = O.transform_all_imu_point(o_i, st[-1], R_il, t_il)
    g_t = L.transformAllImuPoint(g_i, st[-1])
    assert np.allclose(g_t, o_t, **tol)

    # device buffers in and out: the sweep stays in HBM
    d_raw = torch.from_numpy(raw).cuda(); d_rel = torch.from_numpy(rel).cuda(); d_out = torch.zeros_like(d_raw); d_back = torch.zeros_like(d_raw)
    arr = L._imu_states(st)
    R, t = capi.f64(R_il).reshape(9), capi.f64(t_il)
    nw = C.c_int64(0)
    vp = C.c_void_p
    assert capi.lib().srl_distort_frame_by_imu(L.ctx.h, vp(d_raw.data_ptr()), vp(d_rel.data_ptr()), n, C.cast(arr, vp), len(st), t0,
                                               capi.ptr(R), capi.ptr(t), vp(d_out.data_ptr()), C.byref(nw)) == 0
    assert nw.value == n and np.array_equal(d_out.cpu().numpy(), g_i)
    last = L._imu_states([st[-1]])
    assert capi.lib().srl_transform_all_imu_point(L.ctx.h, vp(d_out.data_ptr()), n, C.cast(last, vp), capi.ptr(R), capi.ptr(t), vp(d_back.data_ptr())) == 0
    assert np.array_equal(d_back.cpu().numpy(), g_t)
    assert capi.lib().srl_distort_frame_by_constant(L.ctx.h, vp(d_raw.data_ptr()), vp(d_rel.data_ptr()), n, C.cast(arr, vp), len(st), t0,
                                                    capi.ptr(R), capi.ptr(t), vp(d_out.data_ptr())) == 0
    assert np.array_equal(d_out.cpu().numpy(), g_c)

    # edge cases: empty sweep, a single IMU state, decreasing stamps
    assert L.distortFrameByImu(raw[:0], rel[:0], st, t0)[1] == 0
    assert L.distortFrameByImu(raw[:10], rel[:10], st[:1], t0)[1] == 0
    with pytest.raises(Exception):
        L.distortFrameByImu(raw[:10], rel[:10], [st[1], st[0]], t0)


def test_randomized_parity_many_sweeps_and_poses(L, cfg1_world):
    """A few hundred thousand associations over random sensor poses, sweep patterns and pose errors: every neighbour
    list must equal the oracle's (the FP32 window / guard / fallback logic has to hold on all of them, not on average)."""
    import os
    from sr_livo_b200 import lio
    om, _ = _load_world(L, cfg1_world)
    prm, oprm = lio.r3live_params(max_num_residuals=BIG), O.r3live_params(max_num_residuals=BIG)
    rng = np.random.default_rng(77)
    total = full = 0
    amb0 = L.ctx.counter("fast_ambiguous")
    for trial in range(12):
        pos = (float(rng.uniform(-30, 30)), float(rng.uniform(-8, 8)), float(rng.uniform(1.0, 4.0)))
        sw = synth.make_sweep(20000, seed=2000 + trial, yaw=float(rng.uniform(-3.1, 3.1)), position=pos,
                              pattern="spinning" if trial % 3 == 2 else "livox", dp_max=float(rng.uniform(0.0, 0.3)),
                              dth_max_deg=float(rng.uniform(0.0, 3.0)), pose_seed=trial)
        L.setKeypoints(sw.raw_xyz)
        g = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last, debug=True)
        o = om.build_plane_residuals(sw.raw_xyz, sw.q_init, sw.t_init, sw.t_last, oprm, nthreads=min(32, os.cpu_count() or 1), debug=True)
        _assert_pass_equal(g, o)
        total += sw.raw_xyz.shape[0]
        full += int((o.status >= 1).sum())
    assert total == 240000 and full > 100000
    assert L.ctx.counter("fast_ambiguous") - amb0 <= 0.001 * full


# ---- BASELINE-size properties (size-independent checks; the oracle would take too long to be the checker) ---------
def test_full_size_properties_100k_sweep_large_map():
    from sr_livo_b200 import dist, lio
    L = lio.LioOptimization(max_voxels=1 << 21, sweep_capacity=1 << 17)
    try:
        pts = synth.sample_map_points(400.0, 60.0, seed=2)                 # ~4.5M-point map
        added = L.addPointsToMap(pts)
        nv, npts = L.voxel_map.stats()
        assert added == npts and 3_000_000 < npts < 8_000_000
        assert L.addPointsToMap(pts[:200000]) == 0                          # re-offering stored points adds nothing
        keys, counts, xyz = L.voxel_map.download()
        assert counts.sum() == npts and counts.max() <= 20 and counts.min() >= 1
        assert len({tuple(k) for k in keys.tolist()}) == nv                  # keys unique
        cell = np.trunc(xyz.astype(np.float64)).astype(np.int64)             # every stored point lies in its voxel
        mask = np.arange(20)[None, :] < counts[:, None]
        assert np.all((cell == keys[:, None, :].astype(np.int64))[mask])
        sw = synth.make_sweep(100000, seed=1000, yaw=0.5)
        prm = lio.r3live_params(max_num_residuals=BIG)
        L.setKeypoints(sw.raw_xyz)
        a = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last, debug=True)
        b = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last)
        b2 = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last)
        assert np.array_equal(b.HTH, b2.HTH) and np.array_equal(b.HTh, b2.HTh)             # bitwise, run to run
        assert _close(a.HTH, b.HTH) and a.num_residuals == b.num_residuals                 # debug build of the kernel: to rounding
        assert a.num_residuals <= a.num_full_neighborhoods <= 100000 and a.num_residuals > 50000
        assert np.allclose(a.HTH, a.HTH.T) and np.linalg.eigvalsh(a.HTH).min() > 0
        acc = a.status == 2
        J, h = a.plane[acc, 6:12], a.plane[acc, 13] * a.plane[acc, 14]
        assert np.allclose(a.HTH, J.T @ J, rtol=1e-10) and np.allclose(a.HTh, J.T @ h, rtol=1e-9, atol=1e-9)
        full = a.status >= 1
        assert np.all(np.diff(a.nbr_dist[full], axis=1) >= 0)               # neighbour lists sorted by distance
        assert np.all(np.abs(np.linalg.norm(a.plane[full, 3:6], axis=1) - 1) < 1e-12)
        HTH = np.zeros((6, 6)); res = 0
        for r in range(8):                                                  # 8-way shard sum == whole
            L.sweep.set_shard(*dist.shard_range(100000, r, 8))
            p = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last)
            HTH += p.HTH; res += p.num_residuals
        L.sweep.set_shard(0, 100000)
        assert res == a.num_residuals and np.abs(HTH - a.HTH).max() <= 1e-11 * np.abs(a.HTH).max()
        L.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=synth.prior_covariance())
        summ, fq, ft = L.updateIEKF(prm, sw.t_last)
        assert summ.success and np.linalg.norm(L.eskf_pro.p - sw.t_true) < 0.01
        after = L.buildPlaneResiduals(prm, fq, ft, sw.t_last)
        assert after.loss_sum < 0.2 * a.loss_sum                            # registration reduced the residual
    finally:
        L.close()


def _color_dict(d):
    return {tuple(k): dict(xyz=d["xyz"][i, :c].copy(), rgb=d["rgb"][i, :c].copy(), n_rgb=d["n_rgb"][i, :c].copy(), cov=d["cov"][i, :c].copy(),
                           obs_dist=d["obs_dist"][i, :c].copy(), last_obs=d["last_obs"][i, :c].copy(), last_visited=float(d["last_visited"][i]))
            for i, (k, c) in enumerate(zip(d["keys"].tolist(), d["counts"].tolist()))}


def test_color_map_and_renderer_match_the_oracle(L):
    """Row N4: addPointToColorMap (src/lioOptimization.cpp:448-551, colour branch) and renderPointsInRecentVoxel with
    rgbPoint::updateRgb (src/rgbMapTracker.cpp:181-237, src/cloudMap.cpp:59-101) on the GPU against the sequential oracle:
    voxel contents and order, the fine-cell dedupe that builds rgb_points_vec (order included), the recently-visited voxel
    list (order included), and after two renderings the fused colours, covariances and observation state — all exact."""
    from sr_livo_b200 import capi, lio
    rng = np.random.default_rng(5)
    room = lambda n: np.stack([rng.uniform(-4, 4, n), rng.uniform(-3, 3, n), rng.choice([0.02, 2.4], n) + rng.normal(0, 0.01, n)], axis=1)
    sweep1, sweep2 = room(9000), np.concatenate([room(3000) + [0.4, 0.0, 0.0], room(2000) * [1.0, 1.0, 0.2]])
    cmg = lio.ColorVoxelMap(L.ctx, max_voxels=1 << 12)
    cmo = O.OracleColorMap()
    cam = capi.Camera()
    cam.q_camera_world[:] = [0.01, -0.02, 0.015, 0.9996]          # not normalised on purpose: toRotationMatrix as given
    cam.t_camera_world[:] = [0.1, -0.2, 5.0]
    cam.t_world_camera[:] = [-0.1, 0.2, -5.0]
    cam.fx, cam.fy, cam.cx, cam.cy, cam.fov_margin, cam.cols, cam.rows = 310.0, 305.0, 322.5, 238.25, 0.0001, 640, 480
    cam15 = np.array(list(cam.q_camera_world) + list(cam.t_camera_world) + list(cam.t_world_camera) + [cam.fx, cam.fy, cam.cx, cam.cy, cam.fov_margin])
    try:
        for step, (pts, kw) in enumerate([(sweep1, dict(add_point_step=2, time_sweep_end=1.0, time_last_process=0.0, to_rendering=True)),
                                          (sweep2, dict(add_point_step=1, time_sweep_end=1.1, time_last_process=1.0, to_rendering=True)),
                                          (sweep1[:500] + 0.03, dict(add_point_step=3, time_sweep_end=1.2, time_last_process=1.2, to_rendering=False))]):
            assert cmg.addPoints(pts, **kw) == cmo.add_points(pts, **kw)
            g, o = cmg.download(), cmo.snapshot()
            oc = cmo.counts()
            st = cmg.stats()
            assert (st["voxels"], st["rgb_points"], st["recent"], st["new_recent"]) == (oc["voxels"], oc["rgb_points"], oc["recent"], oc["new_recent"])
            o_rgb_points, o_recent = cmo.lists()
            assert np.array_equal(g["rgb_points"], o_rgb_points)                   # rgb_points_vec: same entries, same order
            assert np.array_equal(g["recent"].astype(np.int32), o_recent)           # voxels_recent_visited: same voxels, same order
            if step < 2:
                img = rng.integers(0, 256, (480, 640, 3), dtype=np.uint8)
                for obs_time in (kw["time_sweep_end"], kw["time_sweep_end"] + 0.05):
                    assert cmg.renderPointsInRecentVoxel(cam, img, obs_time) == cmo.render(cam15, img, obs_time)
                g, o = cmg.download(), cmo.snapshot()
            gd, od = _color_dict(g), _color_dict(o)
            assert gd.keys() == od.keys()
            for k in od:
                for f in ("xyz", "rgb", "n_rgb", "cov", "obs_dist", "last_obs"):
                    assert np.array_equal(gd[k][f], od[k][f]), (step, k, f)
                assert gd[k]["last_visited"] == od[k]["last_visited"]
            if step == 1:
                assert g["n_rgb"].max() >= 3 and (g["rgb"] > 0).any()               # the renderer really coloured points, repeatedly
    finally:
        cmg.close()


def _region_oracle(L, world_pts, margin=3):
    """The oracle map restricted to the voxels around `world_pts` (downloaded from the GPU map, which the product's own
    insert kernel built; byte-equality of that build with the oracle's is the job of the map tests)."""
    keys, counts, xyz = L.voxel_map.download()
    lo = np.floor(world_pts.min(axis=0)).astype(np.int64) - margin
    hi = np.ceil(world_pts.max(axis=0)).astype(np.int64) + margin
    k = keys.astype(np.int64)
    sel = np.all((k >= lo) & (k <= hi), axis=1)
    om = O.OracleMap()
    om.load(keys[sel], counts[sel], xyz[sel])
    return om


@pytest.mark.parametrize("scale", ["cfg2", "cfg5"])
def test_neighbour_ids_bit_exact_at_baseline_scale(scale):
    """BASELINE.json sizes: config 2 (100k-pt Livox sweep, ~10M-pt map) and config 5 (500k-pt spinning sweep, ~50M-pt map).
    The whole sweep runs through the default kernels with per-keypoint outputs; a contiguous-in-space sample of it
    (5k / 20k keypoints) is compared with the oracle on the same map region: status, the 20 neighbour ids in order, the
    neighbour distances (bit-exact), the plane columns (1e-5)."""
    from sr_livo_b200 import lio
    extent, n_pts, pattern, n_sample, max_vox = ((600.0, 100000, "livox", 5000, 1 << 21) if scale == "cfg2"
                                                 else (1340.0, 500000, "spinning", 20000, 1 << 23))
    L = lio.LioOptimization(max_voxels=max_vox, sweep_capacity=n_pts)
    try:
        pts = synth.sample_map_points(extent, 60.0, seed=1)
        L.addPointsToMap(pts)
        del pts
        n_map = L.mapSize()
        assert n_map > (9_000_000 if scale == "cfg2" else 45_000_000)
        sw = synth.make_sweep(n_pts, seed=1000, yaw=0.5, position=(0.0, 3.0, 1.8), pattern=pattern)
        prm = lio.r3live_params(max_num_residuals=BIG)
        L.setKeypoints(sw.raw_xyz)
        g = L.buildPlaneResiduals(prm, sw.q_init, sw.t_init, sw.t_last, debug=True)
        assert g.num_residuals > 0.5 * n_pts
        # the sample: the n_sample keypoints nearest (in the world frame) to a seeded keypoint: a compact map region
        centre = g.world_xyz[12345]
        idx = np.sort(np.argsort(np.linalg.norm(g.world_xyz - centre, axis=1))[:n_sample])
        om = _region_oracle(L, g.world_xyz[idx])
        o = om.build_plane_residuals(sw.raw_xyz[idx], sw.q_init, sw.t_init, sw.t_last, O.r3live_params(max_num_residuals=BIG),
                                     debug=True)
        assert o.num_fragile == 0
        assert np.array_equal(g.status[idx], o.status)
        full = o.status >= 1
        assert full.sum() > 0.5 * n_sample
        assert np.array_equal(g.nbr[idx][full], o.nbr[full])                       # ids, in order: bit-exact
        assert np.array_equal(g.nbr_dist[idx][full], o.nbr_dist[full])
        assert np.array_equal(g.world_xyz[idx], o.world_xyz)
        ref, got = o.plane[full], g.plane[idx][full]
        scale_c = np.maximum(np.abs(ref).max(axis=0), 1e-12)
        assert np.all(np.abs(got - ref) <= REL * scale_c)
    finally:
        L.close()


def test_exact_distance_ties_on_a_lattice_map():
    """Exactly equal distances (the case every other test excludes through the oracle's `fragile` counter).  Map points
    on a 0.25 m lattice in the plane z = 0.125 (all coordinates exact in FP32), keypoints exactly above lattice cell
    centres and lattice nodes, identity pose: many candidates tie bit-for-bit, also at the K-th boundary.
    What holds: the reference keeps, among equal distances, the candidates it visited first (strict `<` at
    src/optimize.cpp:399), and so does the GPU (order (d^2, visit index)): status, the SET of the 20 neighbours and the
    sorted distance list are identical.  What may differ: the ORDER of equal-distance entries inside the list — the
    reference's is whatever std::priority_queue leaves, the GPU's is by visit index — which only permutes the
    accumulation order of the plane fit (vector_neighbors[0] is used for the weight and the plane offset; on this map
    every tied choice gives the same offset and the same distance)."""
    from sr_livo_b200 import lio
    g1 = np.arange(-6.0, 6.0001, 0.25)
    X, Y = np.meshgrid(g1, g1, indexing="ij")
    pts = np.stack([X.ravel(), Y.ravel(), np.full(X.size, 0.125)], axis=1)
    om = O.OracleMap()
    om.add_points(pts, min_distance_points=0.15)
    c1 = np.arange(-3.875, 3.9, 0.25)                       # cell centres: 4 nearest lattice nodes tie, then 8, ...
    n1 = np.arange(-3.75, 3.8, 0.5)                         # lattice nodes: 1 nearest, then 4 tie, 4 tie, ...
    kp = np.concatenate([np.stack(np.meshgrid(c1, c1, indexing="ij"), -1).reshape(-1, 2),
                         np.stack(np.meshgrid(n1, n1, indexing="ij"), -1).reshape(-1, 2)])
    raw = np.concatenate([kp, np.full((kp.shape[0], 1), 0.3125)], axis=1)
    q, t, tl = np.array([0.0, 0.0, 0.0, 1.0]), np.zeros(3), np.array([0.0, 0.0, 5.0])
    L = lio.LioOptimization(max_voxels=1 << 12, sweep_capacity=1 << 12)
    try:
        snap = om.snapshot()
        mp = np.concatenate([x[:c] for c, x in zip(snap[1].tolist(), snap[2])]).astype(np.float64)   # the stored map points
        L.voxel_map.upload(*snap)
        L.setKeypoints(raw)
        for variant in (0, 2):                               # default kernels (with their exact fallback), k1_assoc alone
            L.ctx.set_option("k1_variant", variant)
            g = L.buildPlaneResiduals(lio.r3live_params(max_num_residuals=BIG), q, t, tl, debug=True)
            o = om.build_plane_residuals(raw, q, t, tl, O.r3live_params(max_num_residuals=BIG), debug=True)
            assert o.num_fragile > 0.9 * raw.shape[0]        # the point of this test
            assert np.array_equal(g.status, o.status)
            full = o.status >= 1
            assert full.sum() > 0.9 * raw.shape[0]
            assert np.array_equal(g.nbr_dist[full], o.nbr_dist[full])               # same sorted distances, bit for bit
            code = np.array([1 << 40, 1 << 24, 1 << 8, 1])
            gs = np.sort(g.nbr[full].astype(np.int64) @ code, axis=1)
            os_ = np.sort(o.nbr[full].astype(np.int64) @ code, axis=1)
            # the K-th boundary is tied when the K-th and (K+1)-th smallest squared distances are equal (brute force over the map)
            d2_all = np.sort(((mp[None, :, 0] - raw[full][:, None, 0]) ** 2 + ((mp[None, :, 1] - raw[full][:, None, 1]) ** 2 +
                             (mp[None, :, 2] - raw[full][:, None, 2]) ** 2)), axis=1)
            boundary_tied = d2_all[:, 19] == d2_all[:, 20]
            same_set = np.all(gs == os_, axis=1)
            assert boundary_tied.sum() > 100 and (~boundary_tied).sum() > 100
            assert np.all(same_set[~boundary_tied])       # no tie at the boundary: the neighbour SET is the reference's
            # tie at the boundary: both hold every point closer than the K-th distance and fill up from the tied shell; WHICH
            # tied points survive differs: the reference evicts whatever std::priority_queue has at its top among equal
            # maxima (heap-internal), the GPU keeps the first visited.  Documented deviation, confined to exact FP64 ties.
            for r in np.nonzero(~same_set)[0]:
                dK = np.sqrt(d2_all[r, 19])
                for lst, dist in ((g.nbr[full][r], g.nbr_dist[full][r]), (o.nbr[full][r], o.nbr_dist[full][r])):
                    assert np.all(dist <= dK) and (dist < dK).sum() == (np.sqrt(d2_all[r]) < dK).sum()
            print(f"variant {variant}: boundary ties at {int(boundary_tied.sum())} keypoints, neighbour set differs from the "
                  f"reference heap's at {int((~same_set).sum())} of them")
            same_order = np.all(g.nbr[full] == o.nbr[full], axis=(1, 2))
            print(f"variant {variant}: {int(same_order.sum())} of {int(full.sum())} tied neighbour lists also have the reference's order")
            # GPU order inside a run of equal distances is the reference's visit order (voxel scan order, then index in block)
            d = g.nbr_dist[full]
            nb = g.nbr[full].astype(np.int64)
            vis = ((nb[..., 0] * 64 + nb[..., 1]) * 64 + nb[..., 2]) * 32 + nb[..., 3]     # monotone in (x, y, z, index) for one keypoint
            tie = d[:, 1:] == d[:, :-1]
            assert np.all(vis[:, 1:][tie] > vis[:, :-1][tie])
            # same set (whatever its order) => same plane, weight, residual, Jacobian to rounding
            ref, got = o.plane[full][same_set], g.plane[full][same_set]
            assert np.allclose(got, ref, rtol=REL, atol=1e-9)    # (columns that are exactly 0 in the reference: normal x/y, J_x, J_y)
            assert g.num_residuals == o.num_residuals
    finally:
        L.ctx.set_option("k1_variant", 0)
        L.close()


def test_cpp_adapter_runs_the_update_on_the_gpu(tmp_path, small_world):
    """include/srlivo_b200_lio.hpp driven from a compiled C++ program (the language of the reference): LioBackend
    addPointsToMap / setKeypoints / updateIEKF / optimize on the GPU, results equal to the Python mirror's."""
    import os, subprocess
    from sr_livo_b200 import capi, lio
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sw = small_world["sweep"]
    pts = small_world["pts"]
    P = synth.prior_covariance()
    np.ascontiguousarray(pts, np.float64).tofile(tmp_path / "pts.bin")
    np.ascontiguousarray(sw.raw_xyz, np.float64).tofile(tmp_path / "raw.bin")
    np.concatenate([sw.t_init, sw.q_init, sw.t_last, P.reshape(-1)]).astype(np.float64).tofile(tmp_path / "state.bin")
    src = tmp_path / "drive.cpp"
    src.write_text(r'''
#include <cstdio>
#include <vector>
#include "srlivo_b200_lio.hpp"
static std::vector<double> slurp(const char* path) {
    FILE* f = std::fopen(path, "rb"); std::fseek(f, 0, SEEK_END); long n = std::ftell(f); std::fseek(f, 0, SEEK_SET);
    std::vector<double> v(n / 8); if (std::fread(v.data(), 8, v.size(), f) != v.size()) v.clear(); std::fclose(f); return v;
}
int main(int argc, char** argv) {
    std::string dir = argv[1];
    std::vector<double> pts = slurp((dir + "/pts.bin").c_str()), raw = slurp((dir + "/raw.bin").c_str()), st = slurp((dir + "/state.bin").c_str());
    srl::LioBackend lio(0, nullptr, 1 << 18, 1 << 17);
    long long added = lio.addPointsToMap(pts.data(), pts.size() / 3, 0.15);
    srl_icp_params p; srl_icp_params_r3live(&p); p.max_num_residuals = 2147483647;
    for (int pass = 0; pass < 2; ++pass) {
        std::memset(&lio.eskf, 0, sizeof(lio.eskf));
        for (int i = 0; i < 3; ++i) lio.eskf.p[i] = st[i];
        for (int i = 0; i < 4; ++i) lio.eskf.q[i] = st[3 + i];
        lio.eskf.g[2] = 9.81;
        for (int i = 0; i < 289; ++i) lio.eskf.cov[i] = st[10 + i];
        double fq[4] = {st[3], st[4], st[5], st[6]}, ft[3] = {st[0], st[1], st[2]}, tl[3] = {st[7], st[8], st[9]};
        srl::optimizeSummary s;
        std::vector<double> world(raw.size());
        if (pass == 0) { lio.setKeypoints(raw.data(), raw.size() / 3); s = lio.updateIEKF(p, fq, ft, tl); }
        else s = lio.optimize(raw.data(), raw.size() / 3, p, fq, ft, tl, world.data());
        std::printf("%d %lld %lld %d %d %d %.17g %.17g %.17g %.17g %.17g %.17g %.17g %.17g\n", pass, added, lio.mapSize(), (int)s.success,
                    s.passes_run, s.num_residuals_used, ft[0], ft[1], ft[2], fq[0], fq[1], fq[2], fq[3], pass ? world[3 * 77 + 1] : 0.0);
    }
    lio.enableColorMap(1.0, 20, 1 << 16, 0.15);                              // row N4 through the adapter
    long long stored = lio.addPointsToColorMap(pts.data(), 30000, 2, 1.0, 0.0, true);
    int64_t nv = 0, np = 0, nrgb = 0, nrec = 0, nnew = 0;
    srl_color_map_stats(lio.colorMap(), &nv, &np, &nrgb, &nrec, &nnew);
    std::printf("color %lld %lld %lld %lld %lld\n", stored, (long long)nv, (long long)np, (long long)nrgb, (long long)nrec);
    return 0;
}''')
    exe = tmp_path / "drive"
    libdir = os.path.dirname(capi.LIB_PATH)
    subprocess.check_call(["g++", "-std=c++14", "-O1", "-I", os.path.join(root, "include"), str(src), "-o", str(exe),
                           "-L", libdir, "-lsrlivo_b200", f"-Wl,-rpath,{libdir}"])
    r = subprocess.run([str(exe), str(tmp_path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    rows = [ln.split() for ln in r.stdout.strip().splitlines()]
    assert len(rows) == 3
    cmo = O.OracleColorMap()
    stored = cmo.add_points(pts[:30000], add_point_step=2, time_sweep_end=1.0, time_last_process=0.0, to_rendering=True)
    oc = cmo.counts()
    assert [int(x) for x in rows[2][1:]] == [stored, oc["voxels"], stored, oc["rgb_points"], oc["recent"]]
    rows = rows[:2]
    # the Python mirror on the same inputs
    Lp = lio.LioOptimization(max_voxels=1 << 18, sweep_capacity=1 << 17)
    try:
        added = Lp.addPointsToMap(pts)
        Lp.setKeypoints(sw.raw_xyz)
        Lp.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=P.copy())
        summ, fq, ft = Lp.updateIEKF(lio.r3live_params(max_num_residuals=BIG), sw.t_last)
        for row in rows:
            assert int(row[1]) == added and int(row[2]) == Lp.mapSize() and int(row[3]) == 1
            assert int(row[4]) == summ.passes_run and int(row[5]) == summ.num_residuals_used
            assert np.array_equal(np.array(row[6:9], float), ft) and np.array_equal(np.array(row[9:13], float), fq)   # same library, same bits
        expect = sw.raw_xyz @ O.quat_to_rot(fq).T + ft
        assert abs(float(rows[1][13]) - expect[77, 1]) < 1e-10
    finally:
        Lp.close()


_DIST_WORKER = r"""
import os, sys
sys.path.insert(0, sys.argv[1])
import numpy as np, torch, torch.distributed as tdist
from oracle import oracle_py as O
from sr_livo_b200 import dist, lio, synth
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
tdist.init_process_group("gloo", rank=rank, world_size=world)
dev = rank % torch.cuda.device_count()
pts = synth.sample_map_points(80.0, 60.0, seed=1)
sw = synth.make_sweep(4000, seed=1000, yaw=0.5)
L = lio.LioOptimization(device=dev, max_voxels=1 << 16, sweep_capacity=8192)
L.addPointsToMap(pts)                                   # every rank builds its replica
D = dist.DistributedLio(L, rank, world, native=True)
prm = lio.r3live_params(max_num_residuals=2**31-1)
for rep in range(3):                                    # several updates in a row: sequence numbers / double buffering
    D.set_keypoints(sw.raw_xyz)
    L.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=synth.prior_covariance())
    # last repetition: rank 1 hands every 7th keypoint to the exact kernel, rank 0 none: the two ranks then finish a pass
    # (and run their side of the exchange) in different kernels
    L.ctx.set_option("fast_force_ambiguous_mod", 7 if (rep == 2 and rank == world - 1) else 0)
    out = D.updateIEKF(prm, sw.t_last)
om = O.OracleMap(); om.add_points(pts)
ref = om.update_iekf(sw.raw_xyz, O.Eskf(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=synth.prior_covariance()), sw.t_last,
                     O.r3live_params(max_num_residuals=2**31-1))
assert out["success"] and out["passes"] == ref["passes"], (out["passes"], ref["passes"])
assert np.allclose(out["trace"], ref["trace"], rtol=1e-5, atol=1e-9)
assert np.allclose(L.eskf_pro.p, ref["eskf"].p, atol=1e-9) and np.allclose(L.eskf_pro.q, ref["eskf"].q, atol=1e-9)
t = torch.from_numpy(np.concatenate([L.eskf_pro.p, L.eskf_pro.q, L.eskf_pro.cov.reshape(-1)]))
lst = [torch.zeros_like(t) for _ in range(world)]
tdist.all_gather(lst, t)
assert all(torch.equal(lst[0], x) for x in lst)         # every rank ends bit-identical
# config 3 end to end in C (srl_optimize_host_dist): host buffers in, this rank's rows of the registered sweep out
L.ctx.set_option("fast_force_ambiguous_mod", 0)
L.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=synth.prior_covariance())
world_out = np.full_like(sw.raw_xyz, np.nan)
o2 = D.optimize(sw.raw_xyz, prm, sw.t_last, world_out=world_out)
b, e = o2["range"]
assert (b, e) == dist.shard_range(sw.raw_xyz.shape[0], rank, world) and o2["passes"] == ref["passes"]
assert np.allclose(o2["frame_t"], ref["frame_t"], atol=1e-9) and np.allclose(o2["frame_q"], ref["frame_q"], atol=1e-9)
expect = sw.raw_xyz @ O.quat_to_rot(o2["frame_q"]).T + o2["frame_t"]
assert np.allclose(world_out[b:e], expect[b:e], rtol=0, atol=1e-10)
assert np.isnan(world_out[:b]).all() and np.isnan(world_out[e:]).all()      # only this rank's rows are written
# the baseline without peer memory: one all-reduce of the 32 sums per pass from Python, host-driven loop (native=False)
Db = dist.DistributedLio(L, rank, world, native=False)
Db.set_keypoints(sw.raw_xyz)
L.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=synth.prior_covariance())
ob = Db.updateIEKF(prm, sw.t_last)
assert ob["passes"] == ref["passes"] and np.allclose(ob["frame_t"], o2["frame_t"], atol=1e-9) and np.allclose(ob["frame_q"], o2["frame_q"], atol=1e-9)
D.close(); L.close(); tdist.destroy_process_group()
print("rank", rank, "ok")
"""


@pytest.mark.parametrize("world", [2, 4])
def test_fused_peer_memory_exchange_ranks(tmp_path, world):
    """The sharded update with the exchange fused into the pass's last kernel (CUDA IPC mailboxes) and the ESIKF update
    in each rank's persistent block: `world` processes (one GPU each if the box has them, else sharing GPUs), each owning
    a contiguous range of the keypoints; then the same end to end from host buffers (srl_optimize_host_dist)."""
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "dist_worker.py"
    script.write_text(_DIST_WORKER)
    port = 29700 + (os.getpid() % 1000)
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port + world))
        procs.append(subprocess.Popen([sys.executable, str(script), root], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o[-3000:]


# ---- the CUDA path against the REFERENCE'S OWN CODE (oracle/_ref/libsrl_reference.so, compiled where it lies) ------
# Its outputs on this scene are recorded by tests/test_reference_pin.py (test_small_world_*) in tests/golden/reference_pin.npz.
def _reference_or_skip():
    from oracle import reference_py as Rf
    if not Rf.available():
        pytest.skip("oracle/_ref/libsrl_reference.so was not built: the reference sources are absent")
    return Rf


@pytest.fixture(scope="module")
def ref_pin():
    from refstore import Store
    return Store("reference_pin.npz")


@pytest.mark.parametrize("kw", SMALL_WORLD_PASS)
def test_gpu_pass_equals_the_compiled_reference(L, small_world, ref_pin, kw):
    """One ESIKF pass on the GPU vs lioOptimization::buildPlaneResiduals of the reference's own src/optimize.cpp: transformed
    keypoints bit for bit, the same keypoints accepted in the same order, rows within 1e-5.  The reference's rows are stored as a
    digest: the oracle's rows, which have that digest, stand for them."""
    from refstore import digest, from_near
    from sr_livo_b200 import lio
    r = ref_pin.get(f"small_world.pass{SMALL_WORLD_PASS.index(kw)}")
    om, sw = _load_world(L, small_world)
    o = om.build_plane_residuals(sw.raw_xyz, sw.q_init, sw.t_init, sw.t_last, O.r3live_params(**kw), debug=True)
    rows = o.plane[o.status == 2][:, :15]
    assert r["rows"] == digest(rows)
    ref_world = from_near(r, "world_all", o.world_xyz)
    L.setKeypoints(sw.raw_xyz)
    g = L.buildPlaneResiduals(lio.r3live_params(**kw), sw.q_init, sw.t_init, sw.t_last, debug=True)
    assert not r["threw"] and r["success"] == g.success and r["num_residuals_used"] == g.num_residuals
    visited = g.status >= 0
    assert np.array_equal(g.world_xyz[visited], ref_world[visited])
    got = g.plane[g.status == 2][:, :15]
    assert got.shape == rows.shape
    scale = np.maximum(np.abs(rows).max(axis=0), 1e-12)
    assert np.all(np.abs(got - rows) <= REL * scale)
    assert abs(g.loss_sum - r["loss_sum"]) <= REL * r["loss_sum"]


def test_gpu_update_equals_the_compiled_reference(L, small_world, ref_pin):
    """updateIEKF on the GPU (device-resident loop) vs the reference's own updateIEKF + eskfEstimator::observe: state 1e-5."""
    from sr_livo_b200 import lio
    om, sw = _load_world(L, small_world)
    P = synth.prior_covariance()
    for case, kw in enumerate(SMALL_WORLD_UPDATE):
        r = ref_pin.get(f"small_world.update{case}")
        L.setKeypoints(sw.raw_xyz)
        L.eskf_pro = lio.EskfEstimator(p=sw.t_init.copy(), q=sw.q_init.copy(), v=np.array([0.3, 0.0, 0.0]), cov=P.copy())
        summ, fq, ft = L.updateIEKF(lio.r3live_params(**kw), sw.t_last)
        assert not r["threw"] and summ.success == r["success"] and summ.num_residuals_used == r["num_residuals_used"]
        for f in ("p", "q", "v", "ba", "bg", "g"):
            assert np.allclose(getattr(L.eskf_pro, f), r[f], rtol=REL, atol=1e-9), f
        assert np.allclose(L.eskf_pro.cov, r["cov"], rtol=1e-4, atol=1e-12)
        assert np.allclose(fq, r["frame_q"], atol=1e-9) and np.allclose(ft, r["frame_t"], atol=1e-9)


def test_reference_runs_on_the_gpu_backend(small_world):
    """The maintainer patch of INTEGRATION.md section 2, for real: oracle/_ref/libsrl_reference_gpu.so is the reference's own objects
    with lioOptimization::updateIEKF and ::addPointsToMap replaced at link time by the product's C++ adapter
    (include/srlivo_b200_lio.hpp -> C ABI -> CUDA).  The reference's unmodified optimize() (gridSampling -> updateIEKF ->
    transformPoint) then registers a sweep through its own call sites on the GPU; the result equals the unpatched reference's."""
    Rf = _reference_or_skip()
    if not Rf.available(gpu=True):
        pytest.skip("oracle/_ref/libsrl_reference_gpu.so was not built: the reference sources are absent")
    pts, sw = small_world["pts"], small_world["sweep"]
    ref, rg = Rf.Reference(), Rf.Reference(gpu=True)
    assert ref.add_points_to_map(pts) > 0                       # the reference's own insertion into its host voxelHashMap
    rg.add_points_to_map(pts)                                   # the same call site, patched: the product's insert kernel
    assert rg.gpu_map_is_on_gpu() and rg.num_points() == 0 and rg.gpu_map_points() == ref.num_points()
    P = synth.prior_covariance()
    world0 = synth.registered_points(sw, sw.q_init, sw.t_init)  # point_frame[i].point as the pose prediction left it
    for kw in (dict(max_num_residuals=600), dict(max_num_residuals=BIG)):
        e0 = O.Eskf(p=sw.t_init.copy(), q=sw.q_init.copy(), v=np.array([0.3, 0.0, 0.0]), cov=P.copy())
        r = ref.optimize(world0, sw.raw_xyz, 1.0, e0, sw.t_last, O.r3live_params(**kw))
        g = rg.optimize(world0, sw.raw_xyz, 1.0, e0, sw.t_last, O.r3live_params(**kw))
        assert not g["threw"] and not r["threw"] and g["success"] and r["success"]
        assert g["num_residuals_used"] == r["num_residuals_used"]
        for f in ("p", "q", "v", "ba", "bg", "g"):
            assert np.allclose(getattr(g["eskf"], f), getattr(r["eskf"], f), rtol=REL, atol=1e-9), f
        assert np.allclose(g["eskf"].cov, r["eskf"].cov, rtol=1e-4, atol=1e-12)
        assert np.allclose(g["frame_q"], r["frame_q"], atol=1e-9) and np.allclose(g["frame_t"], r["frame_t"], atol=1e-9)
        assert np.allclose(g["world"], r["world"], rtol=0, atol=1e-6)     # the re-transformed frame (src/optimize.cpp:441-445)
        assert np.linalg.norm(g["eskf"].p - sw.t_true) < 0.02
    reg = synth.registered_points(sw)                            # the registered sweep goes into both maps: streaming through the patch
    ref.add_points_to_map(reg); rg.add_points_to_map(reg)
    assert rg.gpu_map_points() == ref.num_points()
