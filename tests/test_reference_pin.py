"""Pins the oracle restatement (oracle/srl_oracle.cpp) against the REFERENCE'S OWN CODE.

oracle/_ref/libsrl_reference.so holds the reference's src/{optimize,utility,eskfEstimator,cloudMap,state,lioOptimization,
rgbMapTracker,parameters}.cpp compiled unmodified (oracle/Makefile target `reference`), over the stand-in headers of oracle/shim/.
So the left-hand side of every comparison below is produced by the reference's own control flow, containers (tsl::robin_map,
std::tr1::unordered_map, std::priority_queue), member functions, casts and quirks; the right-hand side by the oracle, which the
GPU parity tests use as their checker.

The reference's side is stored in tests/golden/reference_pin.npz (tests/refstore.py): bit-for-bit outputs as digests, the
rest as values.  SRL_RECORD_REFERENCE=1 with the reference libraries built re-runs the reference and rewrites that file.

What stays unpinned: the arithmetic INSIDE Eigen / OpenCV calls (reduction order of small dot products, SelfAdjointEigenSolver,
PartialPivLU, saturating Vec3b operators) — oracle/shim restates it with the same evaluation orders the oracle assumes, so
equality here says nothing about those (DESIGN.md §2).  Everything else that a restatement can get wrong is checked.
"""
import os

import numpy as np
import pytest

from oracle import oracle_py as O
from oracle import reference_py as Rf
from refstore import RECORD, Store, digest, eskf_fields, from_near, map_digest, near
from sr_livo_b200 import synth

BIG = 2 ** 31 - 1
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def sm():
    return np.load(os.path.join(HERE, "golden", "scan_matching.npz"))


@pytest.fixture(scope="module")
def sp():
    return np.load(os.path.join(HERE, "golden", "sweep_prep.npz"))


@pytest.fixture(scope="module")
def ref_out():
    store = Store("reference_pin.npz")
    yield store
    store.save()


def _reference(gpu=False):
    """The reference object, constructed only when its outputs are being recorded."""
    return Rf.Reference(gpu) if RECORD else None


def _pair(sm):
    ref = _reference()
    if ref is not None:
        ref.load(sm["map_keys"], sm["map_counts"], sm["map_xyz"])
    om = O.OracleMap(); om.load(sm["map_keys"], sm["map_counts"], sm["map_xyz"])
    return ref, om


def _tsl():
    return "tsl" in O.backend()


def _as_dict(keys, counts, xyz):
    return {tuple(k): x[:c].copy() for k, c, x in zip(keys.tolist(), counts.tolist(), xyz)}


def _snap(keys, counts, xyz):
    """voxel content (any container order) and the container's iteration order"""
    return dict(map=map_digest(keys, counts, xyz), order=digest(keys, xyz))


def _ref_snap(ref, **kw):
    s = ref.snapshot(**kw)
    return dict(_snap(s["keys"], s["counts"], s["xyz"]), num_points=ref.num_points(), num_voxels=ref.num_voxels())


def _pass_out(r, visited=None):
    """buildPlaneResiduals of the reference: rows and transformed keypoints (of the `visited` ones) as digests"""
    if r["threw"]:
        return dict(threw=True)
    return dict(threw=False, success=r["success"], num_residuals_used=r["num_residuals_used"], loss_sum=r["loss_sum"],
                rows_shape=np.array(r["rows"].shape), rows=r["rows"], world=r["world_xyz"] if visited is None else r["world_xyz"][visited])


PASS_EXACT = ("rows", "world")


def _iekf_out(r):
    return dict(threw=r["threw"], success=r["success"], num_residuals_used=r["num_residuals_used"], frame_q=r["frame_q"],
                frame_t=r["frame_t"], **eskf_fields(r["eskf"]))


def _eskf(r):
    return O.Eskf(**{f: np.asarray(r[f], np.float64).copy() for f in ("p", "q", "v", "ba", "bg", "g", "cov")})


# ---- the reference object itself ----------------------------------------------------------------------------------
def test_reference_constructor_and_hash(ref_out):
    rng = np.random.default_rng(0)
    xyz = [(-1, 2, 3), (0, 0, 0), (-32767, 32767, -1)] + rng.integers(-32767, 32767, (200, 3)).tolist()

    def rec():
        ref = Rf.Reference()
        return dict(laser_point_cov=Rf.lib().ref_laser_point_cov(ref._h), hashes=np.array([Rf.voxel_hash(*v) for v in xyz], np.uint64))
    r = ref_out("constructor_and_hash", rec)
    assert r["laser_point_cov"] == 0.001                                     # src/lioOptimization.cpp:364, what orc_icp_params carries
    assert r["hashes"].tolist() == [O.voxel_hash(*v) for v in xyz]          # std::hash<voxel>, include/cloudMap.h:173-184


# ---- A7 addPointsToMap / addPointToMap, N4 removePointsFarFromLocation -------------------------------------------
@pytest.mark.parametrize("case", [dict(voxel_size=1.0, cap=20, min_dist=0.15, min_num=0), dict(voxel_size=0.5, cap=8, min_dist=0.05, min_num=0),
                                  dict(voxel_size=1.0, cap=20, min_dist=0.0, min_num=0)])
def test_add_points_to_map_equals_the_oracle(ref_out, case):
    rng = np.random.default_rng(11)
    ref = _reference(); om = O.OracleMap()
    tag = "add_points.{voxel_size}_{cap}_{min_dist}".format(**case)
    for sweep in range(4):
        pts = np.concatenate([rng.uniform(-6, 6, (6000, 3)), rng.normal(0, 0.3, (3000, 3)) + [2.2, -1.7, 0.4],
                              np.array([[0.99999999999, 0.1, 0.1], [-0.5, -0.5, -0.5], [0.5, 0.5, 0.5]])])
        a = ref_out(f"{tag}.sweep{sweep}", lambda: dict(added=ref.add_points_to_map(pts, case["voxel_size"], case["cap"], case["min_dist"],
                                                                                     case["min_num"])))["added"]
        b = om.add_points(pts, case["voxel_size"], case["cap"], case["min_dist"], case["min_num"])
        assert a == b
    s = ref_out(f"{tag}.map", lambda: _ref_snap(ref, cap=case["cap"])); o = _snap(*om.snapshot(cap=case["cap"]))
    assert s["num_points"] == om.num_points and s["num_voxels"] == om.num_voxels
    assert s["map"] == o["map"]                                              # same voxels; contents AND order inside every voxel
    if _tsl():                                                               # same container, same insertions: same iteration order
        assert s["order"] == o["order"]
    # min_num_points > 0: only voxels that already hold enough points accept more, unknown voxels are not created (:431,:439)
    more = rng.uniform(-7, 7, (5000, 3))
    a = ref_out(f"{tag}.more", lambda: dict(added=ref.add_points_to_map(more, case["voxel_size"], case["cap"], case["min_dist"], 3)))["added"]
    assert a == om.add_points(more, case["voxel_size"], case["cap"], case["min_dist"], 3)
    assert ref_out(f"{tag}.map_more", lambda: _ref_snap(ref, cap=case["cap"]))["map"] == _snap(*om.snapshot(cap=case["cap"]))["map"]
    # removePointsFarFromLocation (src/lioOptimization.cpp:556-572)
    loc = np.array([1.0, -0.5, 0.2])
    assert ref_out(f"{tag}.remove_far", lambda: dict(removed=ref.remove_far(loc, 4.0)))["removed"] == om.remove_far(loc, 4.0)
    assert ref_out(f"{tag}.map_removed", lambda: _ref_snap(ref, cap=case["cap"]))["map"] == _snap(*om.snapshot(cap=case["cap"]))["map"]


# ---- A3 searchNeighbors ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nb,thr", [(1, 1), (2, 1), (1, 3)])
def test_search_neighbors_equals_the_oracle(ref_out, sm, nb, thr):
    ref, om = _pair(sm)
    blocks = _as_dict(sm["map_keys"], sm["map_counts"], sm["map_xyz"])
    prm = O.r3live_params(max_num_residuals=BIG, frame_id=100 if nb == 1 else 5, threshold_voxel_occupancy=thr)
    o = om.build_plane_residuals(sm["raw_xyz"], sm["q_init"], sm["t_init"], sm["t_last"], prm, debug=True)
    assert o.num_fragile == 0
    idx = np.flatnonzero(o.status >= 0)[::7]
    full = idx[o.status[idx] != 0]

    def rec():
        found = {k: ref.search_neighbors(o.world_xyz[k], nb=nb, size=1.0, K=20, thr=1 if nb == 2 else thr) for k in idx}
        return dict(counts=np.array([found[k][0].shape[0] for k in idx]), xyz=np.concatenate([found[k][0] for k in full]),
                    vox=np.concatenate([found[k][1] for k in full]))
    r = ref_out(f"search_neighbors.nb{nb}_thr{thr}", rec, exact=("xyz", "vox"))
    assert np.all(r["counts"][o.status[idx] == 0] < 20)                     # :78: fewer than min_number_neighbors, keypoint skipped
    assert np.all(r["counts"][o.status[idx] != 0] == 20)
    want = [np.array([blocks[tuple(v[:3])][v[3]] for v in o.nbr[k].tolist()], np.float64) for k in full]
    assert r["xyz"] == digest(np.concatenate(want))                         # same 20 map points, nearest first
    assert r["vox"] == digest(np.concatenate([o.nbr[k][:, :3] for k in full]))
    for k, xyz in zip(full, want):
        d = np.sqrt(((xyz - o.world_xyz[k]) ** 2)[:, 0] + (((xyz - o.world_xyz[k]) ** 2)[:, 1] + ((xyz - o.world_xyz[k]) ** 2)[:, 2]))
        assert np.array_equal(d, o.nbr_dist[k])
    assert full.size > 50


# ---- A2 / A4 buildPlaneResiduals + computeNeighborhoodDistribution ------------------------------------------------
PASS_CASES = {
    "nb1": dict(max_num_residuals=BIG, frame_id=100),
    "nb2_init_frames": dict(max_num_residuals=BIG, frame_id=5),
    "cap100": dict(max_num_residuals=100, frame_id=100),
    "cap600_yaml": dict(max_num_residuals=600, frame_id=100),
    "cap_default_minus1": dict(max_num_residuals=-1, frame_id=100),
    "occupancy3": dict(max_num_residuals=BIG, frame_id=100, threshold_voxel_occupancy=3),
    "gate_tight": dict(max_num_residuals=BIG, frame_id=100, max_dist_to_plane_icp=0.05),
    "weights": dict(max_num_residuals=BIG, frame_id=100, weight_alpha=-0.7, weight_neighborhood=0.4, power_planarity=1.0),
    "too_few": dict(max_num_residuals=BIG, frame_id=100, min_number_neighbors=20, max_dist_to_plane_icp=-1.0),
}


@pytest.mark.parametrize("tag", list(PASS_CASES))
@pytest.mark.parametrize("ext", [False, True])
def test_build_plane_residuals_equals_the_oracle(ref_out, sm, tag, ext):
    ref, om = _pair(sm)
    prm = O.r3live_params(**PASS_CASES[tag])
    R_il = synth.quat_to_rot(synth.quat_from_rotvec([0.02, -0.01, 0.03])) if ext else None
    t_il = np.array([0.05, -0.02, 0.1]) if ext else None
    raw = sm["raw_xyz"] if not ext else (sm["raw_xyz"] - t_il) @ R_il     # same body-frame points through a non-trivial extrinsic
    o = om.build_plane_residuals(raw, sm["q_init"], sm["t_init"], sm["t_last"], prm, R_il, t_il, debug=True)
    visited = o.status >= 0
    r = ref_out(f"pass.{tag}.ext{int(ext)}", lambda: _pass_out(ref.build_plane_residuals(raw, sm["q_init"], sm["t_init"], sm["t_last"], prm,
                                                                                           R_il, t_il), visited), exact=PASS_EXACT)
    assert not r["threw"] and not o.nan_planarity
    assert r["success"] == o.success and r["num_residuals_used"] == o.num_residuals
    assert r["world"] == digest(o.world_xyz[visited])                         # transformKeypoints (:31-42), bit for bit
    rows = o.plane[o.status == 2][:, :15]                                     # accepted keypoints in keypoint order = plane_residuals
    assert tuple(r["rows_shape"]) == rows.shape
    assert r["rows"] == digest(rows)                                          # raw_point, normal, Jacobian, offset, distance, weight: bit for bit
    assert r["loss_sum"] == o.loss_sum
    # the normal equations the oracle hands to the GPU tests are those rows' products (src/optimize.cpp:160-170,235,239)
    if rows.shape[0]:
        J = rows[:, 6:12]; h = rows[:, 13] * rows[:, 14]
        assert np.allclose(J.T @ J, o.HTH, rtol=1e-12, atol=1e-18) and np.allclose(J.T @ h, o.HTh, rtol=1e-11, atol=1e-18)


def test_neighborhood_distribution_on_random_and_degenerate_sets(ref_out, sm):
    ref, om = _pair(sm)
    rng = np.random.default_rng(5)
    sets = []
    for trial in range(200):
        kind = trial % 4
        pts = rng.normal(0, 1, (20, 3)) * ([1, 1, 0.01] if kind == 0 else [1, 0.02, 0.02] if kind == 1 else [1, 1, 1] if kind == 2 else [1, 1, 1e-7])
        sets.append(pts @ synth.quat_to_rot(synth.quat_from_rotvec(rng.normal(0, 1, 3))).T + rng.uniform(-50, 50, 3))
    sets.append(np.tile([[1.0, 2.0, 3.0]], (20, 1)))                         # all points identical

    fields = ("center", "normal", "covariance", "a2D")

    def rec():
        out = [ref.neighborhood(pts) for pts in sets]
        return dict(rc=np.array([rc for rc, _ in out]), **{f: np.stack([nh[f] for _, nh in out[:-1]]) for f in fields})
    r = ref_out("neighborhood", rec, exact=fields)
    want = {f: [] for f in fields}
    for trial, pts in enumerate(sets[:-1]):
        assert r["rc"][trial] == 0
        # against the oracle's eigen restatement (same covariance accumulation order as src/optimize.cpp:327-335)
        bary = np.zeros(3)
        for p in pts:
            bary = bary + p
        bary = bary / 20.0
        cov = np.zeros((3, 3))
        for p in pts:
            for k in range(3):
                for l in range(k, 3):
                    cov[k, l] += (p[k] - bary[k]) * (p[l] - bary[l])
        cov[1, 0], cov[2, 0], cov[2, 1] = cov[0, 1], cov[0, 2], cov[1, 2]
        ev, evec = O.eig3_sym(cov)
        n = evec[:, 0]
        nn = n[0] * n[0] + (n[1] * n[1] + n[2] * n[2])
        n = n / np.sqrt(nn) if nn > 0 else n
        s1, s2, s3 = np.sqrt(abs(ev[2])), np.sqrt(abs(ev[1])), np.sqrt(abs(ev[0]))
        for f, v in zip(fields, (bary, n, cov, (s2 - s3) / s1)):
            want[f].append(v)
    for f in fields:                                                          # every set, bit for bit
        assert r[f] == digest(np.stack(want[f])), f
    # all points identical: 0 / 0 -> NaN planarity -> the reference throws (:348-350)
    assert r["rc"][-1] == 1


def test_nan_planarity_throws_in_both(ref_out, sm):
    # a map whose voxels hold 20 copies of one point each: every neighbourhood is degenerate
    keys = np.array([[0, 0, 0], [1, 0, 0]], np.int16); counts = np.array([20, 20], np.int32)
    xyz = np.zeros((2, 20, 3), np.float32); xyz[0] = [0.5, 0.5, 0.5]; xyz[1] = [1.5, 0.5, 0.5]
    ref = _reference()
    if ref is not None:
        ref.load(keys, counts, xyz)
    om = O.OracleMap(); om.load(keys, counts, xyz)
    raw = np.array([[0.6, 0.5, 0.5]])
    prm = O.r3live_params(max_num_residuals=BIG)
    q, t = np.array([0, 0, 0, 1.0]), np.zeros(3)
    assert ref_out("nan_planarity", lambda: dict(threw=ref.build_plane_residuals(raw, q, t, t, prm)["threw"]))["threw"]
    assert om.build_plane_residuals(raw, q, t, t, prm).nan_planarity


# ---- A1 / A8 updateIEKF + observe ---------------------------------------------------------------------------------
IEKF_CASES = {
    "steady": dict(max_num_residuals=BIG),
    "cap600_yaml": dict(max_num_residuals=600),
    "init_frame_15_iterations": dict(max_num_residuals=BIG, frame_id=5),
    "frame_1_never_converges_early": dict(max_num_residuals=BIG, frame_id=1, init_num_frames=0),
    "loose_thresholds_early_exit": dict(max_num_residuals=BIG, threshold_orientation_norm=5.0, threshold_translation_norm=0.5),
    "one_iteration": dict(max_num_residuals=BIG, num_iters_icp=1),
    "too_few_residuals": dict(max_num_residuals=BIG, max_dist_to_plane_icp=-1.0),
}


def _assert_eskf_equal(a: O.Eskf, b: O.Eskf, rtol, atol):
    for name in ("p", "q", "v", "ba", "bg", "g"):
        assert np.allclose(getattr(a, name), getattr(b, name), rtol=rtol, atol=atol), name
    # (P / c)^-1 is ill-conditioned (c = 0.001, prior entries 1e-5 .. 1): small entries move in their 7th digit between two
    # LU loop orders; measured against the matrix's scale the two covariances agree to 1e-11
    assert np.allclose(a.cov, b.cov, rtol=1e-6, atol=1e-11 * np.abs(b.cov).max())


@pytest.mark.parametrize("tag", list(IEKF_CASES))
def test_update_iekf_equals_the_oracle(ref_out, sm, tag):
    ref, om = _pair(sm)
    prm = O.r3live_params(**IEKF_CASES[tag])
    rng = np.random.default_rng(3)
    e0 = O.Eskf(p=sm["t_init"].copy(), q=sm["q_init"].copy(), v=rng.normal(0, 0.3, 3), ba=rng.normal(0, 0.01, 3), bg=rng.normal(0, 0.001, 3),
                g=np.array([0.03, -0.02, 9.8]), cov=sm["prior_cov"].copy())
    R_il = synth.quat_to_rot(synth.quat_from_rotvec([0.01, 0.02, -0.015])); t_il = np.array([0.04, 0.0, -0.03])
    raw = (sm["raw_xyz"] - t_il) @ R_il
    r = ref_out(f"update_iekf.{tag}", lambda: _iekf_out(ref.update_iekf(raw, e0, sm["t_last"], prm, R_il=R_il, t_il=t_il)))
    o = om.update_iekf(raw, e0, sm["t_last"], prm, R_il=R_il, t_il=t_il)
    assert not r["threw"]
    assert r["success"] == o["success"] and r["num_residuals_used"] == o["num_residuals_used"]
    # the associations are identical pass by pass (previous test), so the two states can only differ by the rounding of the
    # 17-dimensional algebra (Eigen's GEMM / LU loop orders are restated, not pinned): 1e-9
    _assert_eskf_equal(_eskf(r), o["eskf"], rtol=1e-9, atol=1e-11)
    assert np.allclose(r["frame_q"], o["frame_q"], rtol=1e-9, atol=1e-12) and np.allclose(r["frame_t"], o["frame_t"], rtol=1e-9, atol=1e-11)
    if tag == "too_few_residuals":
        assert not r["success"]
        assert np.array_equal(r["p"], e0.p) and np.array_equal(r["cov"], e0.cov)   # early return (:155) leaves the filter untouched
    else:
        assert r["success"] and np.linalg.norm(r["p"] - sm["t_true"]) < np.linalg.norm(e0.p - sm["t_true"])


def test_eskf_observe_equals_the_oracle(ref_out):
    rng = np.random.default_rng(9)
    cases = []
    for trial in range(100):
        q = rng.normal(0, 1, 4); q /= np.linalg.norm(q)
        e = O.Eskf(p=rng.normal(0, 5, 3), q=q, v=rng.normal(0, 1, 3), ba=rng.normal(0, 0.1, 3), bg=rng.normal(0, 0.01, 3),
                   g=np.array([0, 0, 9.81]) + rng.normal(0, 0.2, 3))
        dx = rng.normal(0, 1, 17) * (1e-6 if trial % 3 == 0 else 1e-2 if trial % 3 == 1 else 0.5)   # both branches of so3ToQuat / so3ToRotation
        cases.append((e, dx))
    names = ("p", "q", "v", "ba", "bg", "g")
    r = ref_out("eskf_observe", lambda: {name: np.stack([getattr(Rf.eskf_observe(e, dx), name) for e, dx in cases]) for name in names})
    for trial, (e, dx) in enumerate(cases):
        b = e.observe(dx)
        for name in names:
            assert np.allclose(r[name][trial], getattr(b, name), rtol=1e-14, atol=1e-15), name


# ---- the caller: optimize() = gridSampling -> updateIEKF -> transformPoint (src/optimize.cpp:428-447) -------------
def test_optimize_equals_the_composition_of_oracle_pieces(ref_out, sm):
    ref, om = _pair(sm)
    prm = O.r3live_params(max_num_residuals=600)
    raw = sm["raw_xyz"]
    R0 = synth.quat_to_rot(sm["q_init"])
    world0 = raw @ R0.T + sm["t_init"]                      # point_frame[i].point as the caller left it (pose prediction)
    e0 = O.Eskf(p=sm["t_init"].copy(), q=sm["q_init"].copy(), cov=sm["prior_cov"].copy())
    size = 1.5
    idx = O.grid_sampling(world0, size)
    o = om.update_iekf(raw[idx], e0, sm["t_last"], prm)
    def rec():
        res = ref.optimize(world0, raw, size, e0, sm["t_last"], prm)
        return dict(_iekf_out(res), world=res["world"], grid=Rf.grid_sampling(world0, size), want=Rf.transform_point(raw, o["frame_q"], o["frame_t"]))
    r = ref_out("optimize", rec, exact=("grid",))
    assert r["grid"] == digest(idx)
    assert r["success"] == o["success"] and r["num_residuals_used"] == o["num_residuals_used"]
    _assert_eskf_equal(_eskf(r), o["eskf"], rtol=1e-9, atol=1e-11)
    assert np.allclose(r["world"], r["want"], rtol=0, atol=1e-8)


# ---- N2 gridSampling: the iteration order of std::tr1::unordered_map ------------------------------------------------
@pytest.mark.parametrize("n,size,spread", [(5000, 1.5, 40.0), (20000, 0.8, 60.0), (300, 1.0, 3.0), (1, 1.0, 1.0)])
def test_grid_sampling_order_equals_the_oracle(ref_out, n, size, spread):
    rng = np.random.default_rng(n)
    xyz = rng.uniform(-spread, spread, (n, 3))
    xyz[: n // 10] = xyz[n // 10: 2 * (n // 10)][: n // 10] + 1e-3            # several points per cell: the first one wins
    a = ref_out(f"grid_sampling.{n}", lambda: dict(keep=Rf.grid_sampling(xyz, size)), exact=("keep",))["keep"]
    assert a == digest(O.grid_sampling(xyz, size))


# ---- N3 undistortion / per-point transforms --------------------------------------------------------------------------
def _states(sp):
    return [dict(timestamp=r[0], quat=r[1:5], trans=r[5:8], vel=r[8:11], un_acc=r[11:14], un_gyr=r[14:17]) for r in sp["imu_states"]]


def test_point_transforms_equal_the_oracle(ref_out, sp):
    states = _states(sp)
    raw, rel, t0 = sp["raw"], sp["rel"], float(sp["t0"])
    R_il, t_il = sp["R_il"], sp["t_il"]
    seed_in = np.full_like(raw, -7.0)                                       # points the iterator never reaches keep their value
    rel2 = rel.copy(); rel2[rel.shape[0] // 3] = 1e6
    b, m = O.distort_frame_by_imu(raw, rel, states, t0, R_il, t_il, seed_in)
    b2, m2 = O.distort_frame_by_imu(raw, rel2, states, t0, R_il, t_il, seed_in)
    r = ref_out("point_transforms", lambda: dict(
        by_constant=Rf.distort_frame_by_constant(raw, rel, states, t0, R_il, t_il), by_imu=Rf.distort_frame_by_imu(raw, rel, states, t0, R_il, t_il, seed_in),
        by_imu_cut=Rf.distort_frame_by_imu(raw, rel2, states, t0, R_il, t_il, seed_in), end_frame=Rf.transform_all_imu_point(b2, states[-1], R_il, t_il)),
        exact=("by_constant", "by_imu", "by_imu_cut", "end_frame"))
    assert r["by_constant"] == digest(O.distort_frame_by_constant(raw, rel, states, t0, R_il, t_il))
    assert r["by_imu"] == digest(b) and 0 < m <= raw.shape[0]
    # a point outside every IMU interval stops the one-iterator walk for good (src/utility.cpp:263-308)
    assert r["by_imu_cut"] == digest(b2) and m2 == rel.shape[0] // 3
    assert r["end_frame"] == digest(O.transform_all_imu_point(b2, states[-1], R_il, t_il))


# ---- N4 colour map + renderer -------------------------------------------------------------------------------------------
COLOR_FIELDS = ("counts", "xyz", "rgb", "n_rgb", "cov", "obs_dist", "last_obs", "last_visited")


def _color_snap(s):
    """every field of every colour voxel, voxels by key (the two containers iterate in different orders)"""
    order = np.lexsort(np.asarray(s["keys"]).T[::-1])
    return dict(keys=digest(np.asarray(s["keys"])[order]), **{f: digest(np.asarray(s[f])[order]) for f in COLOR_FIELDS})


def test_color_map_and_renderer_equal_the_oracle(ref_out):
    rng = np.random.default_rng(21)
    ref = _reference()
    oc = O.OracleColorMap(voxel_size=0.5, max_num_points_in_voxel=8, min_distance_points=0.05)
    om = O.OracleMap()
    rows, cols = 96, 128
    fx = fy = 90.0; cx, cy = cols / 2.0, rows / 2.0
    for sweep in range(3):
        pts = np.concatenate([rng.uniform(-2.5, 2.5, (2500, 2)), rng.uniform(3.0, 6.0, (2500, 1))], axis=1)   # in front of the camera
        t_end, t_proc = 10.0 + sweep, 10.0 + sweep - (0.0 if sweep == 1 else 0.5)       # sweep 1: |dt| < 1e-5 -> no voxel becomes recent
        a = ref_out(f"color.sweep{sweep}.add", lambda: dict(added=ref.add_points_to_map(
            pts, 1.0, 20, 0.15, 0, color_voxel_size=0.5, color_max_points=8, color_min_distance=0.05, add_point_step=3,
            time_sweep_end=t_end, time_last_process=t_proc, to_rendering=True)))["added"]
        assert a == om.add_points(pts, 1.0, 20, 0.15, 0)
        oc.add_points(pts, add_point_step=3, time_sweep_end=t_end, time_last_process=t_proc, to_rendering=True)
        ca, cb = ref_out(f"color.sweep{sweep}.counts", lambda: ref.color_counts()), oc.counts()
        assert ca == cb
        la, lb = ref_out(f"color.sweep{sweep}.lists", lambda: dict(zip(("rgb_points", "recent"), ref.color_lists())), exact=("rgb_points", "recent")), oc.lists()
        assert la["rgb_points"] == digest(lb[0]) and la["recent"] == digest(lb[1])  # rgb_points_vec and voxels_recent_visited, in order
        # render twice (first observation, then the fusion branch of updateRgb)
        for k in range(2):
            img = rng.integers(0, 256, (rows, cols, 3), dtype=np.uint8)
            q_cw = synth.quat_from_rotvec(rng.normal(0, 0.02, 3)); t_cw = rng.normal(0, 0.05, 3)
            R = synth.quat_to_rot(q_cw); t_wc = -R.T @ t_cw
            cam = np.concatenate([q_cw, t_cw, t_wc, [fx, fy, cx, cy, 0.005]])
            obs = t_end + 0.01 * (k + 1)
            assert ref_out(f"color.sweep{sweep}.render{k}", lambda: dict(n=ref.color_render(cam, img, obs)))["n"] == oc.render(cam, img, obs)
        sa = ref_out(f"color.sweep{sweep}.map", lambda: _color_snap(ref.snapshot(which=1, cap=8, color=True))); sb = oc.snapshot()
        assert sa == _color_snap(sb)
    assert ca["rgb_points"] > 500 and (sb["n_rgb"] > 1).sum() > 100


# ---- a different, larger scene: several sweeps and poses, map built by the reference's own addPointsToMap -------------
def test_randomized_scene_passes_equal_the_oracle(ref_out):
    pts = synth.sample_map_points(80.0, 40.0, seed=3)
    ref = _reference(); om = O.OracleMap()
    assert ref_out("scene.add", lambda: dict(added=ref.add_points_to_map(pts)))["added"] == om.add_points(pts)
    total = 0
    for i, kw in enumerate([dict(yaw=0.4, position=(0.0, 3.0, 1.8)), dict(yaw=-2.0, position=(6.0, -4.0, 2.2), pattern="spinning"),
                            dict(yaw=1.3, position=(-9.0, 8.0, 1.5), dp_max=0.3, dth_max_deg=3.0)]):
        sw = synth.make_sweep(2500, seed=3100 + i, **kw)
        for frame_id, cap in [(100, BIG), (3, BIG), (100, 600)]:
            prm = O.r3live_params(max_num_residuals=cap, frame_id=frame_id)
            r = ref_out(f"scene.sweep{i}.{frame_id}_{cap}", lambda: _pass_out(ref.build_plane_residuals(sw.raw_xyz, sw.q_init, sw.t_init, sw.t_last, prm)),
                        exact=PASS_EXACT)
            o = om.build_plane_residuals(sw.raw_xyz, sw.q_init, sw.t_init, sw.t_last, prm, debug=True)
            assert o.num_fragile == 0
            assert r["success"] == o.success and r["num_residuals_used"] == o.num_residuals
            assert r["rows"] == digest(o.plane[o.status == 2][:, :15]) and r["loss_sum"] == o.loss_sum
            total += o.num_residuals
    assert total > 5000


# ---- config 4 in miniature: insert, register the next sweep, insert it — all through the reference's member functions --
def test_streaming_insert_then_register_equals_the_oracle(ref_out):
    ref = _reference(); om = O.OracleMap()
    prm = O.r3live_params(max_num_residuals=BIG)
    for i in range(4):
        sw = synth.make_sweep(6000, seed=3300 + i, yaw=0.5, position=(-4.0 + 1.0 * i, 3.0, 1.8))
        if i >= 2:                                                            # the first sweeps only build the map
            e0 = O.Eskf(p=sw.t_init.copy(), q=sw.q_init.copy(), cov=synth.prior_covariance())
            r = ref_out(f"streaming.sweep{i}.update", lambda: _iekf_out(ref.update_iekf(sw.raw_xyz, e0, sw.t_last, prm)))
            o = om.update_iekf(sw.raw_xyz, e0, sw.t_last, prm)
            assert r["success"] and o["success"] and r["num_residuals_used"] == o["num_residuals_used"]
            _assert_eskf_equal(_eskf(r), o["eskf"], rtol=1e-9, atol=1e-11)
            assert np.linalg.norm(r["p"] - sw.t_true) < 0.03
        reg = synth.registered_points(sw)
        assert ref_out(f"streaming.sweep{i}.add", lambda: dict(added=ref.add_points_to_map(reg)))["added"] == om.add_points(reg)
    assert ref_out("streaming.map", lambda: _ref_snap(ref))["map"] == _snap(*om.snapshot())["map"]


def test_many_sweeps_on_host_threads_equal_the_single_calls(ref_out, sm):
    """ref_update_iekf_many (the throughput form bench.py's CPU arm times): every sweep's result equals the single-sweep call, and
    the oracle's update of that sweep."""
    ref, om = _pair(sm)
    prm = O.r3live_params(max_num_residuals=BIG)
    rng = np.random.default_rng(17)
    raws, eskfs, tls = [], [], []
    for s in range(6):
        keep = rng.permutation(sm["raw_xyz"].shape[0])[:400]
        raws.append(sm["raw_xyz"][keep])
        eskfs.append(O.Eskf(p=sm["t_init"] + rng.normal(0, 0.02, 3), q=sm["q_init"].copy(), cov=sm["prior_cov"].copy()))
        tls.append(sm["t_last"])

    def rec():
        ok, out, fq, ft = ref.update_iekf_many(raws, eskfs, tls, prm, n_threads=3)
        one = [ref.update_iekf(raws[s], eskfs[s], tls[s], prm) for s in range(6)]
        return dict(ok=ok, many=digest(*[np.concatenate([e.p, e.cov.ravel(), q]) for e, q in zip(out, fq)]),
                    single=digest(*[np.concatenate([o["eskf"].p, o["eskf"].cov.ravel(), o["frame_q"]]) for o in one]),
                    **{f"{s}.{k}": v for s, o in enumerate(one) for k, v in _iekf_out(o).items()})
    r = ref_out("many_sweeps", rec)
    assert r["ok"] == 6
    assert r["many"] == r["single"]
    for s in range(6):
        o = om.update_iekf(raws[s], eskfs[s], tls[s], prm)
        one = {k.split(".", 1)[1]: v for k, v in r.items() if k.startswith(f"{s}.")}
        assert one["success"] and o["success"] and one["num_residuals_used"] == o["num_residuals_used"]
        _assert_eskf_equal(_eskf(one), o["eskf"], rtol=1e-9, atol=1e-11)


# ---- a 1.6M-point map (the bench's world, 240 m side) and a sample of a 100k-point sweep: the scale the GPU id tests run at
def test_mid_scale_sample_equals_the_oracle(ref_out):
    pts = synth.sample_map_points(240.0, 60.0, seed=1)
    om = O.OracleMap(); om.add_points(pts)
    del pts
    ref = _reference()
    if ref is not None:
        ref.load(*om.snapshot())
    assert ref_out("mid_scale.map", lambda: dict(num_points=ref.num_points()))["num_points"] == om.num_points > 1_500_000
    sw = synth.make_sweep(100000, seed=1000, yaw=0.5)
    pick = np.random.default_rng(1).permutation(100000)[:6000]
    raw = sw.raw_xyz[pick]
    prm = O.r3live_params(max_num_residuals=BIG)
    r = ref_out("mid_scale.pass", lambda: _pass_out(ref.build_plane_residuals(raw, sw.q_init, sw.t_init, sw.t_last, prm)), exact=PASS_EXACT)
    o = om.build_plane_residuals(raw, sw.q_init, sw.t_init, sw.t_last, prm, debug=True)
    assert o.num_fragile == 0 and r["num_residuals_used"] == o.num_residuals > 4000
    assert r["rows"] == digest(o.plane[o.status == 2][:, :15]) and r["world"] == digest(o.world_xyz)


# ---- the one unpinned choice that reaches a discrete outcome: the order of a 3-term reduction inside Eigen ------------------
def test_no_discrete_outcome_depends_on_the_order_of_three_term_reductions(ref_out, sm):
    """oracle/_ref/libsrl_reference_packet.so = the same reference sources over the stand-in with dot / norm / product rows of three
    terms evaluated as (c0 + c1) + c2 (what a vectorised Eigen 3.3 most likely does for plain Vector3d operands) instead of
    c0 + (c1 + c2) (what the oracle, the default stand-in and the CUDA kernels do).  Transformed keypoints and distances move by an
    ulp; the accepted keypoints, their 20 neighbours (same map points, same order) and the final pose do not change on any scene.
    Stored: the default build's outputs (checked against the oracle) and how far the other build's moved from them."""
    scenes = [(sm["map_keys"], sm["map_counts"], sm["map_xyz"], sm["raw_xyz"], sm["q_init"], sm["t_init"], sm["t_last"])]
    om = O.OracleMap(); om.add_points(synth.sample_map_points(80.0, 40.0, seed=3))
    sw = synth.make_sweep(3000, seed=3100, yaw=0.4)
    scenes.append((*om.snapshot(), sw.raw_xyz, sw.q_init, sw.t_init, sw.t_last))
    moved = 0
    for si, (keys, counts, xyz, raw, q, t, tl) in enumerate(scenes):
        a, b = _reference(), _reference("packet")
        if RECORD:
            a.load(keys, counts, xyz); b.load(keys, counts, xyz)
        oa = O.OracleMap(); oa.load(keys, counts, xyz)
        for j, kw in enumerate((dict(max_num_residuals=BIG), dict(max_num_residuals=BIG, frame_id=5), dict(max_num_residuals=600))):
            prm = O.r3live_params(**kw)
            o = oa.build_plane_residuals(raw, q, t, tl, prm, debug=True)
            rows_o = o.plane[o.status == 2][:, :15]

            def rec():
                ra, rb = a.build_plane_residuals(raw, q, t, tl, prm), b.build_plane_residuals(raw, q, t, tl, prm)
                close = rb["rows"].shape == ra["rows"].shape and np.allclose(ra["rows"], rb["rows"], rtol=1e-11, atol=1e-13)
                return dict(num_a=ra["num_residuals_used"], num_b=rb["num_residuals_used"], rows_a=ra["rows"], rows_shape_b=np.array(rb["rows"].shape),
                            keypoints_b=rb["rows"][:, 0:3], rows_close=close, world_a=ra["world_xyz"][o.status >= 0], world_maxdiff=np.abs(ra["world_xyz"] - rb["world_xyz"]).max(),
                            moved=int((ra["world_xyz"] != rb["world_xyz"]).sum()))
            r = ref_out(f"packet.scene{si}.{j}", rec, exact=("rows_a", "keypoints_b", "world_a"))
            assert r["rows_a"] == digest(rows_o) and r["num_a"] == o.num_residuals                # the default build: the oracle's rows
            assert r["world_a"] == digest(o.world_xyz[o.status >= 0])                               # and transformed keypoints
            assert r["num_a"] == r["num_b"] and tuple(r["rows_shape_b"]) == rows_o.shape
            assert r["keypoints_b"] == digest(rows_o[:, 0:3])                                      # the same keypoints were accepted, in order
            assert r["rows_close"]                                                                 # rows within rtol 1e-11, atol 1e-13
            assert r["world_maxdiff"] < 1e-13
            moved += r["moved"]

        def rec_nbr():                                                                            # at the last case's keypoints
            wa, wb = a.build_plane_residuals(raw, q, t, tl, prm)["world_xyz"], b.build_plane_residuals(raw, q, t, tl, prm)["world_xyz"]
            la = [a.search_neighbors(wa[k]) for k in range(0, raw.shape[0], 5)]
            lb = [b.search_neighbors(wb[k]) for k in range(0, raw.shape[0], 5)]
            return dict(a=digest(*[x for pair in la for x in pair]), b=digest(*[x for pair in lb for x in pair]), full=sum(x.shape[0] == 20 for x, _ in la))
        nbr = ref_out(f"packet.scene{si}.neighbours", rec_nbr)
        assert nbr["a"] == nbr["b"]                                                               # neighbour lists: identical map points, identical order
        assert nbr["full"] > 50
        e0 = O.Eskf(p=t.copy(), q=q.copy(), cov=synth.prior_covariance())
        u = ref_out(f"packet.scene{si}.update", lambda: dict(**{f"a.{k}": v for k, v in _iekf_out(a.update_iekf(raw, e0, tl, O.r3live_params(max_num_residuals=BIG))).items()},
                                                             **{f"b.{k}": v for k, v in _iekf_out(b.update_iekf(raw, e0, tl, O.r3live_params(max_num_residuals=BIG))).items()}))
        assert u["a.success"] and u["b.success"] and u["a.num_residuals_used"] == u["b.num_residuals_used"]
        assert np.allclose(u["a.p"], u["b.p"], rtol=0, atol=1e-11) and np.allclose(u["a.q"], u["b.q"], rtol=0, atol=1e-12)
    assert moved > 100          # the two orders do differ in the last place — the test is not vacuous


# ---- exact distance ties and keypoints on cell boundaries: the heap's behaviour among equal distances is the reference's own ----
def test_exact_ties_and_cell_boundaries_equal_the_oracle(ref_out):
    g = np.arange(-2.0, 4.0, 0.25)
    lattice = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    lattice = lattice[np.random.default_rng(2).permutation(lattice.shape[0])]
    ref = _reference(); om = O.OracleMap()
    assert ref_out("ties.add", lambda: dict(added=ref.add_points_to_map(lattice, 1.0, 20, 0.15, 0)))["added"] == om.add_points(lattice, 1.0, 20, 0.15, 0)
    s = ref_out("ties.map", lambda: _ref_snap(ref)); k, c, x = om.snapshot()
    assert s["order"] == _snap(k, c, x)["order"] if _tsl() else True
    # keypoints on lattice points, on cell faces / edges / corners (exact integers), at cell centres, and on the doubled cell 0
    kp = np.concatenate([lattice[:300], np.stack(np.meshgrid([-1.0, 0.0, 1.0, 2.0], [0.0, 1.0, 0.5], [1.0, 1.5, -0.0], indexing="ij"), -1).reshape(-1, 3),
                         np.array([[0.999999999999, 0.5, 0.5], [-0.999999999999, 0.5, 0.5], [1e-300, -1e-300, 0.5]])])
    q, t = np.array([0.0, 0.0, 0.0, 1.0]), np.zeros(3)
    for j, kw in enumerate((dict(max_num_residuals=BIG), dict(max_num_residuals=BIG, frame_id=5), dict(max_num_residuals=BIG, max_dist_to_plane_icp=10.0))):
        prm = O.r3live_params(**kw)
        r = ref_out(f"ties.pass{j}", lambda: _pass_out(ref.build_plane_residuals(kp, q, t, np.array([-5.0, 0.3, 0.2]), prm)), exact=PASS_EXACT)
        o = om.build_plane_residuals(kp, q, t, np.array([-5.0, 0.3, 0.2]), prm, debug=True)
        assert o.num_fragile > 100                                            # ties and boundaries everywhere: exactly what the other tests exclude
        if r["threw"]:
            assert o.nan_planarity
            continue
        assert r["num_residuals_used"] == o.num_residuals and r["world"] == digest(o.world_xyz)
        assert r["rows"] == digest(o.plane[o.status == 2][:, :15])
    blocks = _as_dict(k, c, x)
    o = om.build_plane_residuals(kp, q, t, np.array([-5.0, 0.3, 0.2]), O.r3live_params(max_num_residuals=BIG), debug=True)
    full = [i for i in range(0, kp.shape[0], 3) if o.status[i] >= 1]      # the neighbour lists themselves, ties included
    r = ref_out("ties.neighbours", lambda: dict(zip(("xyz", "vox"), map(np.concatenate, zip(*[ref.search_neighbors(kp[i]) for i in full])))),
                exact=("xyz", "vox"))
    want = [np.array([blocks[tuple(v[:3])][v[3]] for v in o.nbr[i].tolist()], np.float64) for i in full]
    assert r["xyz"] == digest(np.concatenate(want)) and r["vox"] == digest(np.concatenate([o.nbr[i][:, :3] for i in full]))


# ---- the caller of the path: stateEstimation over a stream (src/lioOptimization.cpp:983-1035) ------------------------------------------
def _rel_pose(q0, t0, q, t):
    """pose (q, t) expressed in the frame of pose (q0, t0)"""
    R0 = synth.quat_to_rot(q0)
    q0_inv = np.array([-q0[0], -q0[1], -q0[2], q0[3]])
    return synth._quat_mul_xyzw(q0_inv, q), R0.T @ (t - t0)


def _transform(raw, q, t):
    """raw points in the world frame of pose (q, t), by the oracle's transformKeypoints (an empty map: nothing else runs)"""
    return O.OracleMap().build_plane_residuals(raw, q, t, t, O.r3live_params(max_num_residuals=BIG), debug=True).world_xyz


def test_state_estimation_stream_equals_the_composition_of_oracle_pieces(ref_out):
    """Seven sweeps through the reference's own stateEstimation — frame 1 only fills the map, frames 2-3 run with the init-frame
    parameters (nb = 2, >= 15 iterations, init_sample_voxel_size), the rest with the steady ones — against gridSampling -> updateIEKF ->
    transformPoint -> addPointsToMap composed from the oracle's pieces with the same per-frame switches (the Python the GPU tests use)."""
    n_frames, init_num_frames, n = 7, 4, 5000
    sweeps = [synth.make_sweep(n, seed=3500 + i, yaw=0.2, position=(0.05 * i, 3.0, 1.8), dp_max=0.03, dth_max_deg=0.3) for i in range(n_frames)]
    q0, t0 = sweeps[0].q_true, sweeps[0].t_true
    ref = _reference()
    if ref is not None:
        ref.stream_reset()
    om = O.OracleMap()
    P = synth.prior_covariance()
    t_prev = None
    for k, sw in enumerate(sweeps, start=1):
        if k <= 2:
            q_pred, t_pred = np.array([0.0, 0.0, 0.0, 1.0]), np.zeros(3)        # stateInitialization: identity for the first two frames
        else:
            q_pred, t_pred = _rel_pose(q0, t0, sw.q_init, sw.t_init)            # a perturbed prediction in the frame of sweep 0
        e0 = O.Eskf(p=t_pred.copy(), q=q_pred.copy(), cov=P.copy())
        prm = O.r3live_params(frame_id=k, init_num_frames=init_num_frames)      # yaml cap 600

        def rec():
            res = ref.stream_push(sw.raw_xyz, k, q_pred, t_pred, e0, prm, init_num_frames=init_num_frames)
            out = dict(_iekf_out(res), num_points=ref.num_points(), **near("world", res["world"], _transform(sw.raw_xyz, res["frame_q"], res["frame_t"])))
            if k > 2:
                out.update(near("world_pred", Rf.transform_point(sw.raw_xyz, q_pred, t_pred), _transform(sw.raw_xyz, q_pred, t_pred)))
            return out
        r = ref_out(f"stream.frame{k}", rec)
        r_world = from_near(r, "world", _transform(sw.raw_xyz, r["frame_q"], r["frame_t"]))
        assert not r["threw"] and r["success"]
        # the same step from the oracle's pieces
        if k > 1:
            world_pred = sw.raw_xyz if k <= 2 else from_near(r, "world_pred", _transform(sw.raw_xyz, q_pred, t_pred))
            idx = O.grid_sampling(world_pred, 1.0 if k < init_num_frames else 1.5)
            o = om.update_iekf(sw.raw_xyz[idx], e0, t_prev, prm, frame_q=q_pred, frame_t=t_pred)
            assert o["success"] and o["num_residuals_used"] == r["num_residuals_used"]
            assert o["passes"] >= (2 if k >= init_num_frames else 2)
            _assert_eskf_equal(_eskf(r), o["eskf"], rtol=1e-9, atol=1e-11)
            assert np.allclose(r["frame_q"], o["frame_q"], atol=1e-11) and np.allclose(r["frame_t"], o["frame_t"], atol=1e-11)
            world = ref_out(f"stream.frame{k}.transform", lambda: near("world", Rf.transform_point(sw.raw_xyz, o["frame_q"], o["frame_t"]),
                                                                         _transform(sw.raw_xyz, o["frame_q"], o["frame_t"])))
            world = from_near(world, "world", _transform(sw.raw_xyz, o["frame_q"], o["frame_t"]))
            assert np.allclose(r_world, world, rtol=0, atol=1e-9)
            t_prev = o["frame_t"].copy()
            if k > 2:                                                            # registration pulls the perturbed prediction back to the truth
                q_true, t_true = _rel_pose(q0, t0, sw.q_true, sw.t_true)
                assert np.linalg.norm(o["frame_t"] - t_true) < 0.02
        else:
            world = sw.raw_xyz.copy()                                            # frame 1: identity, no optimisation (:1010-1019)
            assert np.array_equal(r_world, world) and np.array_equal(r["frame_t"], np.zeros(3))
            t_prev = np.zeros(3)
        om.add_points(r_world, 1.0, 20, 0.1, 0)                                  # odometryOptions::min_distance_points = 0.1
        assert r["num_points"] == om.num_points
    assert ref_out("stream.map", lambda: _ref_snap(ref))["map"] == _snap(*om.snapshot())["map"]


def test_threaded_oracle_port_equals_the_compiled_reference(ref_out, sm):
    """The form of the oracle bench.py times on all host threads (keypoint ranges over std::threads, private sums, fixed-order combine)
    against the single-threaded reference: same residuals, state to 1e-9."""
    ref, om = _pair(sm)
    prm = O.r3live_params(max_num_residuals=BIG)
    e0 = O.Eskf(p=sm["t_init"].copy(), q=sm["q_init"].copy(), cov=sm["prior_cov"].copy())
    r = ref_out("threaded_port", lambda: _iekf_out(ref.update_iekf(sm["raw_xyz"], e0, sm["t_last"], prm)))
    for nt in (2, 5, 8):
        o = om.update_iekf(sm["raw_xyz"], e0, sm["t_last"], prm, nthreads=nt)
        assert o["success"] and o["num_residuals_used"] == r["num_residuals_used"]
        _assert_eskf_equal(_eskf(r), o["eskf"], rtol=1e-9, atol=1e-11)


# ---- a seeded sweep over the parameter space (icpOptions the yaml files never set included) --------------------------------------------
def test_random_parameter_sets_equal_the_oracle(ref_out):
    rng = np.random.default_rng(77)
    pts = synth.sample_map_points(80.0, 50.0, seed=9)
    sw = synth.make_sweep(1500, seed=3700, yaw=-0.7, position=(2.0, -3.0, 1.6))
    maps = {}
    checked = 0
    for trial in range(36):
        size = [0.5, 1.0, 2.0][trial % 3]
        cap = [20, 8, 32][(trial // 3) % 3]
        if (size, cap) not in maps:
            ref = _reference(); om = O.OracleMap()
            added = ref_out(f"random_params.map_{size}_{cap}", lambda: dict(added=ref.add_points_to_map(pts, size, cap, 0.07 * size, 0)))["added"]
            assert added == om.add_points(pts, size, cap, 0.07 * size, 0)
            maps[(size, cap)] = (ref, om)
        ref, om = maps[(size, cap)]
        kmax = int(rng.choice([5, 10, 20, 30]))
        kw = dict(size_voxel_map=size, max_number_neighbors=kmax, min_number_neighbors=int(rng.integers(3, kmax + 1)),
                  threshold_voxel_occupancy=int(rng.choice([1, 2, 5])), voxel_neighborhood=int(rng.choice([0, 1, 2])),
                  power_planarity=float(rng.choice([0.5, 1.0, 2.0, 3.0])), max_dist_to_plane_icp=float(rng.choice([0.05, 0.3, 1.0])),
                  weight_alpha=float(rng.uniform(-1, 1)), weight_neighborhood=float(rng.uniform(0.05, 1)),
                  max_num_residuals=int(rng.choice([BIG, 600, 50, -1])), frame_id=int(rng.choice([1, 5, 19, 20, 100])),
                  init_num_frames=int(rng.choice([0, 20])))
        prm = O.r3live_params(**kw)
        dq = synth.quat_from_rotvec(rng.normal(0, 0.01, 3))
        q = synth.quat_mul(sw.q_true, dq); t = sw.t_true + rng.normal(0, 0.05, 3)
        r = ref_out(f"random_params.{trial}", lambda: _pass_out(ref.build_plane_residuals(sw.raw_xyz, q, t, sw.t_last, prm)), exact=PASS_EXACT)
        o = om.build_plane_residuals(sw.raw_xyz, q, t, sw.t_last, prm, debug=True)
        assert r["threw"] == bool(o.nan_planarity), kw
        if r["threw"]:
            continue
        assert r["success"] == o.success and r["num_residuals_used"] == o.num_residuals, kw
        assert r["rows"] == digest(o.plane[o.status == 2][:, :15]), kw
        assert r["loss_sum"] == o.loss_sum
        checked += r["rows_shape"][0]
    assert checked > 5000


def test_random_update_parameter_sets_equal_the_oracle(ref_out, sm):
    ref, om = _pair(sm)
    rng = np.random.default_rng(78)
    n_ok = 0
    for trial in range(16):
        kw = dict(max_num_residuals=int(rng.choice([BIG, 600, 200])), num_iters_icp=int(rng.choice([1, 2, 5, 8])),
                  threshold_translation_norm=float(rng.choice([0.0, 0.001, 0.01, 0.2])), threshold_orientation_norm=float(rng.choice([0.0, 0.01, 0.1, 2.0])),
                  frame_id=int(rng.choice([1, 2, 5, 100])), init_num_frames=int(rng.choice([0, 20])), laser_point_cov=float(rng.choice([0.001, 0.01, 0.0001])),
                  max_dist_to_plane_icp=float(rng.choice([0.1, 0.3])), power_planarity=float(rng.choice([1.0, 2.0])))
        prm = O.r3live_params(**kw)
        e0 = O.Eskf(p=sm["t_init"] + rng.normal(0, 0.03, 3), q=synth.quat_mul(sm["q_init"], synth.quat_from_rotvec(rng.normal(0, 0.004, 3))),
                    v=rng.normal(0, 0.5, 3), ba=rng.normal(0, 0.02, 3), bg=rng.normal(0, 0.002, 3), g=np.array([0.0, 0.0, 9.81]) + rng.normal(0, 0.05, 3),
                    cov=sm["prior_cov"] * float(rng.choice([0.1, 1.0, 10.0])))
        r = ref_out(f"random_update.{trial}", lambda: _iekf_out(ref.update_iekf(sm["raw_xyz"], e0, sm["t_last"], prm)))
        o = om.update_iekf(sm["raw_xyz"], e0, sm["t_last"], prm)
        assert not r["threw"] and r["success"] == o["success"] and r["num_residuals_used"] == o["num_residuals_used"], kw
        _assert_eskf_equal(_eskf(r), o["eskf"], rtol=1e-8, atol=1e-10)
        assert np.allclose(r["frame_q"], o["frame_q"], atol=1e-10) and np.allclose(r["frame_t"], o["frame_t"], atol=1e-10), kw
        n_ok += r["success"]
    assert n_ok >= 12


# ---- the scene of the GPU tests that compare the CUDA path with the compiled reference (tests/test_gpu_parity.py reads these) ----
SMALL_WORLD_PASS = [dict(max_num_residuals=BIG), dict(max_num_residuals=BIG, frame_id=5), dict(max_num_residuals=600)]
SMALL_WORLD_UPDATE = [dict(max_num_residuals=BIG), dict(max_num_residuals=600)]


@pytest.mark.parametrize("case", range(len(SMALL_WORLD_PASS)))
def test_small_world_pass_equals_the_oracle(ref_out, small_world, case):
    om, sw = small_world["omap"], small_world["sweep"]
    prm = O.r3live_params(**SMALL_WORLD_PASS[case])
    o = om.build_plane_residuals(sw.raw_xyz, sw.q_init, sw.t_init, sw.t_last, prm, debug=True)

    def rec():
        ref = Rf.Reference()
        ref.load(*om.snapshot())
        res = ref.build_plane_residuals(sw.raw_xyz, sw.q_init, sw.t_init, sw.t_last, prm)
        return dict(_pass_out(res, o.status >= 0), **near("world_all", res["world_xyz"], o.world_xyz))
    r = ref_out(f"small_world.pass{case}", rec, exact=PASS_EXACT)
    assert not r["threw"] and r["success"] == o.success and r["num_residuals_used"] == o.num_residuals
    assert r["world"] == digest(o.world_xyz[o.status >= 0])
    assert r["rows"] == digest(o.plane[o.status == 2][:, :15]) and r["loss_sum"] == o.loss_sum
    from_near(r, "world_all", o.world_xyz)


@pytest.mark.parametrize("case", range(len(SMALL_WORLD_UPDATE)))
def test_small_world_update_equals_the_oracle(ref_out, small_world, case):
    om, sw = small_world["omap"], small_world["sweep"]
    prm = O.r3live_params(**SMALL_WORLD_UPDATE[case])
    e0 = O.Eskf(p=sw.t_init.copy(), q=sw.q_init.copy(), v=np.array([0.3, 0.0, 0.0]), cov=synth.prior_covariance())

    def rec():
        ref = Rf.Reference()
        ref.load(*om.snapshot())
        return _iekf_out(ref.update_iekf(sw.raw_xyz, e0, sw.t_last, prm))
    r = ref_out(f"small_world.update{case}", rec)
    o = om.update_iekf(sw.raw_xyz, e0, sw.t_last, prm)
    assert not r["threw"] and r["success"] == o["success"] and r["num_residuals_used"] == o["num_residuals_used"]
    _assert_eskf_equal(_eskf(r), o["eskf"], rtol=1e-9, atol=1e-11)
