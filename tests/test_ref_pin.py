"""PINS THE ORACLE AGAINST THE REFERENCE'S OWN SOURCE (CPU).

oracle/_ref/libvxref.so is the reference's hot-path code itself — the original project's VoxelSLAM/src/{tools,preintegration,voxel_map,loop_refine}.hpp
compiled unmodified (oracle/Makefile, `ref` target) against stand-ins for the absent third-party headers (oracle/ref_standin/: an eager
mini-Eigen restating Eigen 3.3.7's published kernels, PCL / ROS / GTSAM declarations).  Every check below runs the SAME seeded inputs through
that library (ref_api) and through the hand-written restatement (oracle_api) that the GPU parity tests compare against, so the restatement's
control flow, constants and formulas are anchored in the reference's real code; the tolerance left over is Eigen-internal summation order.
Also pins the harness's IMU stand-in (tests/harness/synth.hpp) against the real IMU_PRE.

The reference side of each comparison comes from the `ref` fixture (tests/ref_golden.py): what the library computed on these inputs is stored under
tests/golden/ref_pin/ — small quantities whole, the bit-exact ones of large arrays as digests, the toleranced ones of large arrays as a seeded row
sample — so the tests run in any checkout.  tests/golden/make_ref_pin_golden.py records it again from the library (`ref.ra` is that library while
recording and None otherwise)."""
import json
import os

import numpy as np
import pytest

import oracle_api as oa
import ref_api
import ref_golden
import scenes
import synth
import voxel_slam_b200 as vx
from ref_golden import digest

HERE = os.path.dirname(os.path.abspath(__file__))
ORDER = ["x", "y", "z", "layer", "path"]


@pytest.fixture
def ref(request):
    """the reference build's side of this test: computed by the library and stored while recording, read back otherwise"""
    record = ref_golden.recording()
    if record and not ref_api.available():
        pytest.fail("recording needs oracle/_ref/libvxref.so (make -C oracle ref)")
    rec = ref_golden.Recording(request.node.name, record, ref_api)
    yield rec
    rec.finish()


def relinf(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(np.max(np.abs(b)), 1e-300))


def relinf_rows(R, b):
    """relinf over the sampled rows R of the reference's array against the same rows of b, scaled by all of b"""
    b = np.asarray(b)
    assert R.n == len(b)
    return float(np.max(np.abs(R.rows - b[R.idx])) / max(np.max(np.abs(b)), 1e-300))


def test_keys_and_hash_bit_exact(ref):
    ra = ref.ra
    cases = json.load(open(os.path.join(HERE, "golden", "voxel_keys.json")))
    for vs in sorted({c["voxel_size"] for c in cases}):
        sub = [c for c in cases if c["voxel_size"] == vs]
        p = np.array([[float.fromhex(h) for h in c["p"]] for c in sub])
        k = ref.value(f"golden_cases_{vs}", lambda: dict(zip(("xyz", "hash"), ra.voxel_keys(p, vs))))      # the reference's cut_voxel + std::hash<VOXEL_LOC>
        assert k["xyz"].tolist() == [c["key"] for c in sub]
        assert [int(v) for v in k["hash"]] == [int(c["hash"]) for c in sub]
    rng = np.random.default_rng(7)
    p = np.concatenate([rng.uniform(-500, 500, (20000, 3)), np.round(rng.uniform(-50, 50, (2000, 3))), rng.uniform(-1e-6, 1e-6, (500, 3)), rng.uniform(-3e7, 3e7, (500, 3))])
    for vs in (0.3, 1.0, 2.0, 15.0):
        b, hb = oa.voxel_keys(p, vs)
        assert ref.digest(f"keys_{vs}", lambda: ra.voxel_keys(p, vs)) == digest(b, hb)


def test_eigensolver_qr_vs_jacobi(ref):
    """Eigen's tridiagonal-QR (stand-in restatement of SelfAdjointEigenSolver::compute) vs the oracle's cyclic Jacobi vs LAPACK."""
    rng = np.random.default_rng(3)
    As = []
    for t in range(400):
        if t % 2 == 0:                                     # thin plane far from the origin: cov = P/N - c c^T with heavy cancellation
            n = rng.standard_normal(3); n /= np.linalg.norm(n)
            pts = rng.uniform(-0.5, 0.5, (50, 3)); pts -= np.outer(pts @ n, n) * (1 - 0.01)
            pts += rng.uniform(-100, 100, 3)
            As.append(np.cov(pts.T, bias=True))
        else:
            B = rng.standard_normal((3, 3)); As.append(B @ B.T * 10 ** rng.uniform(-6, 3))
    r = ref.value("eig3", lambda: dict(zip(("w", "U"), map(np.array, zip(*[ref.ra.eig3(A) for A in As])))))
    worst = 0.0
    for A, wr, Ur in zip(As, r["w"], r["U"]):
        wo, Uo = oa.eig3(A)
        wn = np.linalg.eigvalsh(A)
        s = max(abs(wn).max(), 1e-300)
        assert np.max(np.abs(wr - wn)) < 1e-13 * s and np.max(np.abs(wo - wn)) < 1e-13 * s
        worst = max(worst, np.max(np.abs(wr - wo)) / s)
        assert np.allclose(Ur @ Ur.T, np.eye(3), atol=1e-13)
        for k in range(3):
            gap = min(abs(wn[k] - wn[j]) for j in range(3) if j != k) / s
            if gap > 1e-4:
                assert abs(abs(Ur[:, k] @ Uo[:, k]) - 1) < 1e-9 / gap * 1e-4 + 1e-12
    assert worst < 1e-14


def test_point_cluster_and_exp(ref):
    ra = ref.ra
    rng = np.random.default_rng(5)
    pts = rng.uniform(-30, 30, (500, 3))
    assert ref.digest("cluster", lambda: ra.cluster_from_points(pts)) == digest(oa.cluster_from_points(pts))     # same operations in the same order: bit-exact
    c = oa.cluster_from_points(pts)
    poses = [synth.perturb_pose(synth.true_pose(20.0, i), 99 + i, 0.3, 5.0) for i in range(20)]
    a = ref.value("cluster_transform", lambda: np.array([ra.cluster_transform(c, pose) for pose in poses]))
    for ai, pose in zip(a, poses):
        b = oa.cluster_transform(c, pose)
        assert np.max(np.abs(ai - b) / (np.abs(b) + 1e-9)) < 1e-14
    ws = ([0, 0, 0], [1e-12, 0, 0], [1e-11, 2e-11, 0], [0.3, -0.2, 0.9], [3.0, 0.1, -0.2])
    e = ref.value("so3_exp", lambda: np.array([ra.so3_exp(w) for w in ws]))
    for ei, w in zip(e, ws):
        assert np.max(np.abs(ei - oa.so3_exp(w))) < 1e-16 + 1e-15


@pytest.mark.parametrize("W,pts,L", [(5, 4000, 6.0), (10, 8000, 10.0)])
def test_factor_residual_hessian_and_lidar_ba(W, pts, L, ref):
    ra = ref.ra
    sc = scenes.make_window(W=W, pts_per_scan=pts, L=L, seed=3)
    of = sc["oracle_factor"]
    rf = ra and ra.OracleFactor.from_dense(W, sc["clusters10"], sc["fix10"], None, sc["eig12"], sc["sum10"])
    assert ref.value("size", lambda: rf.size()) == of.size()
    # acc_evaluate2 with the map-time cache
    Hr, Jr, rr = rf.hessian(sc["poses_est"]) if ra else (None, None, None)
    Ho, Jo, ro = of.hessian(sc["poses_est"])
    r = ref.value("hessian", lambda: {"J": Jr, "r": rr})
    assert abs(r["r"] - ro) <= 1e-15 * abs(ro) and relinf(r["J"], Jo) < 1e-12 and relinf_rows(ref.rows("hessian_H", lambda: Hr), Ho) < 1e-12
    Hb = ra and Hr.reshape(W, 6, W, 6)
    assert ref.value("hessian_mirrored", lambda: all(np.array_equal(Hb[i, :, j, :], Hb[j, :, i, :].T) for i in range(W) for j in range(i)))   # lower block triangle mirrored (voxel_map.hpp:237-239)
    # evaluate_only_residual + the cache it leaves behind
    # sum of lambda_0: every lambda_0 (~1e-4) carries the eigensolvers' 1e-16 * lambda_max (QR here, Jacobi in the restatement)
    assert abs(ref.value("residual_true", lambda: rf.residual(sc["poses_true"])) - of.residual(sc["poses_true"])) < 1e-11 * abs(ro)
    er, eo = rf and rf.export(), of.export()
    assert relinf_rows(ref.rows("sum10", lambda: er["sum10"]), eo["sum10"]) < 1e-14
    L3 = ref.rows("lambda", lambda: er["eig12"][:, :3])
    lo = eo["eig12"][L3.idx, :3]
    assert L3.n == len(eo["eig12"]) and np.max(np.abs(L3.rows - lo) / np.max(np.abs(lo), axis=1, keepdims=True)) < 1e-9
    # Lidar_BA_Optimizer::damping_iter, thread split included
    for iters, thd in ((4, 2), (3, 1)):
        a = ra and ra.OracleFactor.from_dense(W, sc["clusters10"], sc["fix10"], None, sc["eig12"], sc["sum10"]).lidar_ba(sc["poses_est"], max_iter=iters, thd_num=thd)
        b = oa.OracleFactor.from_dense(W, sc["clusters10"], sc["fix10"], None, sc["eig12"], sc["sum10"]).lidar_ba(sc["poses_est"], max_iter=iters, thd_num=thd)
        av = ref.value(f"lidar_ba_{iters}_{thd}", lambda: {k: a[k] for k in ("poses", "resis", "is_converge")})
        inc = np.max(np.abs(b["poses"] - sc["poses_est"]))
        assert np.max(np.abs(av["poses"] - b["poses"])) < 1e-8 * inc
        assert relinf_rows(ref.rows(f"lidar_ba_{iters}_{thd}_hess", lambda: a["hess"]), b["hess"]) < 1e-10
        assert relinf(av["resis"], b["resis"]) < 1e-11 and av["is_converge"] == b["is_converge"]


def test_too_few_voxels_is_the_reference_exit_path(ref):
    ra = ref.ra
    sc = scenes.make_window(W=5, pts_per_scan=3000, L=6.0, seed=2)
    status = ref.value("status", lambda: ra.OracleFactor.from_dense(5, sc["clusters10"][:1], sc["fix10"][:1], None, sc["eig12"][:1], sc["sum10"][:1])
                       .lidar_ba(sc["poses_est"], max_iter=2, thd_num=2)["status"])
    assert status == -3


def test_imu_standin_matches_real_imu_pre(ref):
    """tests/harness/synth.hpp ImuPre (what bench.py and the GPU tests hand to vxs_li_ba) vs the reference's IMU_PRE on the same samples."""
    W = 8
    tr = np.stack([synth.true_pose(8.0, i) for i in range(W)])
    st = scenes.states_from_poses(np.stack([synth.perturb_pose(tr[i], 50 + i, 2e-3, 1e-2) for i in range(W)]))
    st[:, 12:15] += 0.02 * np.random.default_rng(0).standard_normal((W, 3))
    st[:, 15:21] += 1e-3 * np.random.default_rng(1).standard_normal((W, 6))
    a, b = ref.ra and ref.ra.RefImuWindow(tr), synth.ImuWindow(tr)
    for g in (False, True):
        ev = a and a.eval(st, with_gravity=g)
        r = ref.value(f"eval_{g}", lambda: {"c": ev[0], "g": ev[2]})
        ca, ga = r["c"], r["g"]
        cb, Bb, gb = b.eval(st, with_gravity=g)
        assert abs(ca - cb) < 1e-9 * abs(cb) and relinf_rows(ref.rows(f"eval_{g}_B", lambda: ev[1]), Bb) < 1e-9 and relinf(ga, gb) < 1e-9


@pytest.mark.parametrize("gravity,iters", [(False, 3), (True, 3), (True, 5)])
def test_li_ba_against_the_reference_optimizers(gravity, iters, ref):
    ra = ref.ra
    W = 8
    sc = scenes.make_window(W=W, pts_per_scan=6000, L=8.0, seed=13)
    st = scenes.states_from_poses(sc["poses_est"])
    st[:, 12:15] += 0.02 * np.random.default_rng(0).standard_normal((W, 3))
    rf = ra and ra.OracleFactor.from_dense(W, sc["clusters10"], sc["fix10"], None, sc["eig12"], sc["sum10"])
    of = oa.OracleFactor.from_dense(W, sc["clusters10"], sc["fix10"], None, sc["eig12"], sc["sum10"])
    a = rf and rf.li_ba(st, ra.RefImuWindow(sc["poses_true"]), with_gravity=gravity, max_iter=iters)      # LI_BA_Optimizer(+Gravity)::damping_iter + IMU_PRE
    b = of.li_ba(st, synth.ImuWindow(sc["poses_true"]), with_gravity=gravity, max_iter=iters)           # restatement + harness IMU stand-in
    av = ref.value("li_ba", lambda: {"states": a["states"], "resis": a["resis"]})
    inc = np.max(np.abs(b["states"] - st))
    assert np.max(np.abs(av["states"] - b["states"])) < 1e-6 * inc
    assert relinf_rows(ref.rows("hess", lambda: a["hess"]), b["hess"]) < 1e-8
    if gravity:
        assert relinf(av["resis"], b["resis"]) < 1e-9
    ea, eb = rf and rf.export(), of.export()                                                              # cache left for OctoTree::margi
    assert relinf_rows(ref.rows("sum10", lambda: ea["sum10"]), eb["sum10"]) < 1e-9


def compare_factor_sets(ref, tag, ea, eb, tol=1e-12):
    """ea: the reference build's export (None unless recording), eb: the oracle's; both are put in voxel-id order"""
    if ea is not None:
        pa = np.argsort(ea["ids"], order=ORDER)
        ea = {k: ea[k][pa] for k in ("ids", "clusters10", "sum10", "fix10", "eig12")}
    pb = np.argsort(eb["ids"], order=ORDER)
    eb = {k: eb[k][pb] for k in ("ids", "clusters10", "sum10", "fix10", "eig12")}
    C = ref.rows(f"{tag}.clusters10", lambda: ea["clusters10"])
    assert C.n == len(eb["ids"])
    assert ref.digest(f"{tag}.ids", lambda: ea["ids"]) == digest(eb["ids"])
    assert ref.digest(f"{tag}.counts", lambda: ea["clusters10"][:, :, 9]) == digest(eb["clusters10"][:, :, 9])       # bit-exact point-to-(voxel, frame) assignment
    cb = eb["clusters10"][C.idx]
    assert np.max(np.abs(C.rows - cb) / (np.abs(cb) + 1e-6)) < tol
    for k in ("sum10", "fix10"):
        R = ref.rows(f"{tag}.{k}", lambda: ea[k])
        assert np.max(np.abs(R.rows - eb[k][R.idx]) / (np.abs(eb[k][R.idx]) + 1e-6)) < tol
    L3 = ref.rows(f"{tag}.lambda", lambda: ea["eig12"][:, :3])
    lb = eb["eig12"][L3.idx, :3]
    assert np.max(np.abs(L3.rows - lb) / np.max(np.abs(lb), axis=1, keepdims=True)) < 1e-12


def compare_gba_sets(ref, tag, ga, gb, clusters=False):
    """OctreeGBA keeps no identity: voxels are matched by their (exactly equal) point counts and centroids"""
    key = lambda g: np.lexsort(np.round(g["sum10"][:, [8, 7, 6, 9]], 6).T)
    if ga is not None:
        ka = key(ga)
        ga = {k: ga[k][ka] for k in ("sum10", "clusters10")}
    kb = key(gb)
    gb = {k: gb[k][kb] for k in ("sum10", "clusters10")}
    S = ref.rows(f"{tag}.sum10", lambda: ga["sum10"])
    assert S.n == len(gb["sum10"])
    assert ref.digest(f"{tag}.counts", lambda: ga["clusters10"][:, :, 9]) == digest(gb["clusters10"][:, :, 9])
    assert np.max(np.abs(S.rows - gb["sum10"][S.idx]) / (np.abs(gb["sum10"][S.idx]) + 1e-6)) < 1e-12
    if clusters:
        C = ref.rows(f"{tag}.clusters10", lambda: ga["clusters10"])
        cb = gb["clusters10"][C.idx]
        assert np.max(np.abs(C.rows - cb) / (np.abs(cb) + 1e-6)) < 1e-12
    return S.n


@pytest.mark.parametrize("W,pts,L,ml", [(5, 6000, 6.0, 2), (4, 20000, 14.0, 2), (3, 5000, 6.0, 0), (6, 3000, 5.0, 3)])
def test_window_map_build(W, pts, L, ml, ref):
    """cut_voxel + OctoTree::recut + tras_opt (the reference's motion_init sequence) vs the restatement: identical voxel set and assignment."""
    ra = ref.ra
    tr, est = scenes.poses_true_est(W, L, 11)
    p, off = scenes.make_points(W, pts, L, 11, tr)
    mp = vx.MapParams.make(voxel_size=1.0, max_layer=ml)
    a, b = ra and ra.build_window_factor(mp, p, off, est), oa.build_window_factor(mp, p, off, est)
    assert ref.value("size", lambda: a.size()) == b.size() > 20
    compare_factor_sets(ref, "plain", a and a.export(), b.export())
    # fixed map points + a shifted scene (negative coordinates, a plane on a cell face)
    sh = np.array([-7.37, -3.37, -0.37])
    est2 = est.copy(); est2[:, 9:] += sh
    fix = (p[: pts // 2] @ tr[0, :9].reshape(3, 3).T + tr[0, 9:]) + sh
    a, b = ra and ra.build_window_factor(mp, p, off, est2, fix_pts=fix), oa.build_window_factor(mp, p, off, est2, fix_pts=fix)
    assert ref.value("size_shifted", lambda: a.size()) == b.size() > 20
    compare_factor_sets(ref, "shifted", a and a.export(), b.export())


@pytest.mark.parametrize("vs,me,thre,minp,ml", [(0.5, 0.0025, (0.25, 0.25, 0.25, 0.25), (5, 5, 5, 5), 2), (2.0, 0.01, (0.1, 0.15, 0.2, 0.3), (20, 12, 8, 5), 3),
                                                (1.0, 0.001, (1 / 16.0, 1 / 9.0, 1 / 4.0, 1.0), (30, 20, 10, 5), 2), (1.5, 0.05, (0.5, 0.5, 0.5, 0.5), (5, 5, 5, 5), 1)])
def test_window_map_build_nondefault_parameters(vs, me, thre, minp, ml, ref):
    """The same sequence under parameter sets away from the launch-file defaults: voxel size, min_eigen_value, per-layer plane thresholds
    (plane_eigen_value_thre, already inverted as voxelslam.cpp:825 leaves them) and per-layer min_point — every branch of plane_judge / recut keyed on them."""
    ra = ref.ra
    W, pts, L = 5, 8000, 9.0
    tr, est = scenes.poses_true_est(W, L, 23)
    p, off = scenes.make_points(W, pts, L, 23, tr)
    mp = vx.MapParams.make(voxel_size=vs, min_eigen_value=me, plane_thre=thre, min_point=tuple(float(x) for x in minp), max_layer=ml)
    a, b = ra and ra.build_window_factor(mp, p, off, est), oa.build_window_factor(mp, p, off, est)
    assert ref.value("size", lambda: a.size()) == b.size() > 5
    compare_factor_sets(ref, "window", a and a.export(), b.export())
    ga, gb = ra and ra.build_gba_factor(mp, p.astype(np.float32), off, est, threads=2).export(), oa.build_gba_factor(mp, p.astype(np.float32), off, est, threads=2).export()
    assert compare_gba_sets(ref, "gba", ga, gb) > 5


def test_ragged_and_empty_scans(ref):
    """Edge cases of the map builds and the down-sampling: scans of very different sizes, an EMPTY scan and a one-point scan inside the window; empty and
    one-point clouds through down_sampling_voxel."""
    ra = ref.ra
    W, L = 6, 7.0
    tr, est = scenes.poses_true_est(W, L, 31)
    sizes = [5000, 0, 1, 7000, 37, 2500]
    scans = [synth.gen_scan(L, i, max(n, 1), tr[i], seed=0x5EED0000 + 31)[:n] for i, n in enumerate(sizes)]
    p = np.concatenate(scans); off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    mp = vx.MapParams.make(voxel_size=1.0, max_layer=2)
    a, b = ra and ra.build_window_factor(mp, p, off, est), oa.build_window_factor(mp, p, off, est)
    assert ref.value("size", lambda: a.size()) == b.size() > 50
    eb = b.export()
    compare_factor_sets(ref, "window", a and a.export(), eb)
    assert np.all(eb["clusters10"][:, 1, 9] == 0) and np.sum(eb["clusters10"][:, 2, 9]) <= 1            # the empty scan observes nothing, the one-point scan at most one voxel
    ga, gb = ra and ra.build_gba_factor(mp, p.astype(np.float32), off, est, threads=2).export(), oa.build_gba_factor(mp, p.astype(np.float32), off, est, threads=2).export()
    assert compare_gba_sets(ref, "gba", ga, gb) > 50
    for name, cloud in (("empty", np.zeros((0, 3), dtype=np.float32)), ("one", np.array([[1.25, -2.5, 0.75]], dtype=np.float32))):
        da, db = ref.value(f"ds_{name}", lambda: {k: v for k, v in ra.down_sampling(cloud, 0.5).items() if k in ("xyz", "count")}), oa.down_sampling(cloud, 0.5)
        assert len(da["xyz"]) == len(db["xyz"]) == len(cloud) and np.array_equal(da["xyz"], db["xyz"]) and np.array_equal(da["count"], db["count"])


def test_gba_map_build(ref):
    ra = ref.ra
    W = 6
    tr, est = scenes.poses_true_est(W, 8.0, 41, rot_sigma=3e-3, pos_sigma=2e-2)
    xyz, off = scenes.make_points(W, 3000, 8.0, 41, tr, dtype=np.float32)
    for vs, me in ((2.0, 0.1), (1.0, 0.0025)):
        mp = vx.MapParams.make(voxel_size=vs, min_eigen_value=me, max_layer=2)
        for thd in (1, 2):
            ea, eb = ra and ra.build_gba_factor(mp, xyz, off, est, threads=thd).export(), oa.build_gba_factor(mp, xyz, off, est, threads=thd).export()
            assert compare_gba_sets(ref, f"vs{vs}_thd{thd}", ea, eb, clusters=True) > 10


def test_down_sampling(ref):
    ra = ref.ra
    rng = np.random.default_rng(8)
    pts = np.concatenate([rng.uniform(-20, 20, (30000, 3)), np.round(rng.uniform(-5, 5, (500, 3)))]).astype(np.float32)
    for vs in (0.25, 1.0):
        for close in (False, True):
            a, b = ra and ra.down_sampling(pts, vs, close=close), oa.down_sampling(pts, vs, close=close)
            ia, ib = a and np.argsort(a["index"]), np.argsort(b["index"])
            assert ref.digest(f"index_{vs}_{close}", lambda: a["index"][ia]) == digest(b["index"][ib])                      # same cells (identified by their first / picked point)
            assert ref.digest(f"xyz_{vs}_{close}", lambda: a["xyz"][ia].view(np.uint32)) == digest(b["xyz"][ib].view(np.uint32))    # float running mean, bit-exact
            if not close:
                assert ref.digest(f"count_{vs}", lambda: a["count"][ia]) == digest(b["count"][ib])
    assert ref.value("too_fine_is_none", lambda: ra.down_sampling(pts, 0.0005) is None)
    pv = np.concatenate([rng.uniform(-20, 20, (20000, 3)), rng.uniform(0, 1e-3, (20000, 9))], axis=1)
    a, b = ra and ra.down_sampling_pvec(pv, 0.5), oa.down_sampling_pvec(pv, 0.5)
    ka, kb = a and np.lexsort(a["xyz"].T), np.lexsort(b["xyz"].T)
    assert ref.digest("pvec", lambda: (a["xyz"][ka].view(np.uint32), a["var_diag"][ka].view(np.uint32))) == digest(b["xyz"][kb].view(np.uint32), b["var_diag"][kb].view(np.uint32))


def _plane_rows(pl, k, extra):
    """per plane, in the order k: center (3), normal (3), plane_var (36), pl[extra] (1)"""
    return np.concatenate([pl["center"][k], pl["normal"][k], pl["plane_var"][k].reshape(-1, 36), pl[extra][k][:, None]], axis=1)


def _flip_by_normal(rows_a, rows_b):
    """plane_var of b with cov(n, c) flipped where b's normal has the opposite sign of a's"""
    sgn = np.sign(np.sum(rows_a[:, 3:6] * rows_b[:, 3:6], axis=1))
    Vb = rows_b[:, 6:42].reshape(-1, 6, 6).copy()
    Vb[:, :3, 3:] *= sgn[:, None, None]; Vb[:, 3:, :3] *= sgn[:, None, None]
    return Vb


def test_margi_plane_update_and_match(ref):
    """OctoTree::margi + plane_update (incl. the cov_add by-product of push) + match + the EKF accumulation loop."""
    ra = ref.ra
    W, L = 4, 6.0
    tr, est = scenes.poses_true_est(W, L, 5)
    pts, off = scenes.make_points(W, 6000, L, 5, tr)
    mp = vx.MapParams.make(voxel_size=1.0, max_layer=2)
    a, b = ra and ra.LocalMap(mp, pts, off, tr, 1e-4, mgsize=1), oa.LocalMap(mp, pts, off, tr, 1e-4, mgsize=1)
    pa, pb = a and a.planes(), b.planes()
    ka, kb = pa and np.lexsort(np.round(pa["voxel_center"], 9).T), np.lexsort(np.round(pb["voxel_center"], 9).T)
    P = ref.rows("planes", lambda: _plane_rows(pa, ka, "radius"))
    assert P.n == len(pb["N"]) > 20
    assert ref.digest("plane_cells", lambda: (pa["voxel_center"][ka], pa["half"][ka], pa["N"][ka])) == digest(pb["voxel_center"][kb], pb["half"][kb], pb["N"][kb])
    Pb = _plane_rows(pb, kb, "radius")[P.idx]
    Pa = P.rows
    assert np.max(np.abs(Pa[:, :3] - Pb[:, :3])) < 1e-13
    assert np.max(np.abs(np.abs(np.sum(Pa[:, 3:6] * Pb[:, 3:6], axis=1)) - 1)) < 1e-9          # normals up to sign
    Va, Vb = Pa[:, 6:42].reshape(-1, 6, 6), _flip_by_normal(Pa, Pb)                              # cov(n, c) flips with the sign of n
    assert np.max(np.abs(Va - Vb) / (np.max(np.abs(Vb), axis=(1, 2), keepdims=True))) < 1e-6
    assert np.array_equal(Pa[:, 42], Pb[:, 42]) or np.max(np.abs(Pa[:, 42] - Pb[:, 42]) / Pb[:, 42]) < 1e-6
    # odometry association of a new scan: match flags bit-exact, sums 1e-9
    pose = synth.perturb_pose(tr[W - 1], 77, 1e-3, 5e-3)
    scan = synth.gen_scan(L, W - 1, 4000, tr[W - 1], seed=0x5EED0000 + 5)
    pv = np.zeros((scan.shape[0], 12)); pv[:, :3] = scan; pv[:, [3, 7, 11]] = 1e-4
    rv, tv = np.eye(3) * 1e-6, np.eye(3) * 1e-5
    for passes in (1, 2):
        oa_ = a and a.odom_accumulate(pv, pose, rv, tv, passes=passes)
        ob_ = b.odom_accumulate(pv, pose, rv, tv, passes=passes)
        o = ref.value(f"odom_{passes}", lambda: {k: oa_[k] for k in ("n", "HTH", "HTz", "nnt")})
        assert o["n"] == ob_["n"] > 500 and ref.digest(f"odom_{passes}_flags", lambda: oa_["flags"]) == digest(ob_["flags"])
        assert relinf(o["HTH"], ob_["HTH"]) < 1e-9 and relinf(o["HTz"], ob_["HTz"]) < 1e-9 and relinf(o["nnt"], ob_["nnt"]) < 1e-9


def _leaf_key(s):
    return np.lexsort(np.concatenate([np.round(s["voxel_center"], 9), s["layer"][:, None]], axis=1).T)


def _compare_sliding_state(ref, i, sa, sb, exact_fields, tol):
    """one scan of the sliding-window sequence: window bookkeeping, the leaves' exact fields and point counts, a sample of their clusters"""
    ka = sa and _leaf_key(sa)
    kb = _leaf_key(sb)
    w = ref.value(f"s{i}.window", lambda: {k: sa[k] for k in ("win_count", "win_base", "ring", "poses")})
    assert w["win_count"] == sb["win_count"] and w["win_base"] == sb["win_base"] and np.array_equal(w["ring"], sb["ring"])
    exact = lambda s, k: tuple(s[f][k] for f in exact_fields) + (s["opt_state"][k] >= 0,) + tuple(s[f][k][..., 9] for f in ("pcr_add", "pcr_fix", "slots"))
    assert ref.digest(f"s{i}.leaves", lambda: exact(sa, ka)) == digest(*exact(sb, kb)), i
    clusters = lambda s, k: np.concatenate([s["pcr_add"][k], s["pcr_fix"][k], s["slots"][k].reshape(len(k), -1)], axis=1)
    R = ref.rows(f"s{i}.clusters", lambda: clusters(sa, ka))
    assert R.n == len(kb)
    y = clusters(sb, kb)[R.idx]
    assert np.max(np.abs(R.rows - y) / (np.abs(y) + 1e-6)) < tol, i
    return w


def test_sliding_window_map_sequence(ref):
    """voxelslam.cpp:1599-1712 map side over 14 scans with a 5-scan window: after EVERY scan the two implementations hold the same leaves with the
    same slot clusters, fix clusters, plane flags, opt_state and ring."""
    ra = ref.ra
    Wn, L, nscan = 5, 6.0, 14
    mp = vx.MapParams.make(voxel_size=1.0, max_layer=2)
    a, b = ra and ra.SlidingSim(mp, Wn, 1, max_points=100), oa.SlidingSim(mp, Wn, 1, max_points=100)
    for i in range(nscan):
        pose = synth.true_pose(L, i)
        est = synth.perturb_pose(pose, 700 + i, 1e-3, 5e-3) if i else pose
        scan = synth.gen_scan(L, i, 3000, pose, seed=0x5EED0000 + 21)
        if ra:
            a.add_scan(scan, est)
        b.add_scan(scan, est)
        sa, sb = a and a.state(), b.state()
        w = _compare_sliding_state(ref, i, sa, sb, ("voxel_center", "half", "layer", "is_plane", "isexist", "has_sw", "in_slide", "last_num", "n_point_fix"), 1e-11)
        assert np.array_equal(w["poses"], sb["poses"])
    assert sb["win_base"] == nscan - Wn + 1 and ref.value("n_fix", lambda: int(np.sum(sa["pcr_fix"][:, 9] > 0))) > 10       # scans were marginalised into pcr_fix


def _pv_records(scan, seed):
    """pointVar records with a full (symmetric positive) per-point variance, as pvec_update leaves them"""
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((scan.shape[0], 3, 3)) * 0.01
    var = A @ np.transpose(A, (0, 2, 1)) + np.eye(3) * 1e-5
    return np.concatenate([scan, var.reshape(-1, 9)], axis=1)


def test_sliding_window_with_ba_between_recut_and_margi(ref):
    """The loop as the reference runs it: per scan cut + recut + tras_opt, then (window full) a BA that moves x_buf and overwrites the factor cache,
    then margi reads pcr_add / eig back from the factor (opt_state path) — reference build vs restatement, plus the plane table and one odometry pass."""
    ra = ref.ra
    Wn, L, nscan = 6, 6.0, 16
    mp = vx.MapParams.make(voxel_size=1.0, max_layer=2)
    a, b = ra and ra.SlidingSim(mp, Wn, 1, max_points=60), oa.SlidingSim(mp, Wn, 1, max_points=60)
    for i in range(nscan):
        pose = synth.true_pose(L, i)
        est = synth.perturb_pose(pose, 900 + i, 2e-3, 1e-2) if i else pose
        pv = _pv_records(synth.gen_scan(L, i, 2500, pose, seed=0x5EED0000 + 33), i)
        if ra:
            a.add_scan_pv(pv, est, ba_iters=2)
        b.add_scan_pv(pv, est, ba_iters=2)
        sa, sb = a and a.state(), b.state()
        w = _compare_sliding_state(ref, i, sa, sb, ("voxel_center", "layer", "is_plane", "isexist", "has_sw", "in_slide", "last_num", "n_point_fix"), 1e-8)
        assert np.max(np.abs(w["poses"] - sb["poses"])) < 1e-9                                   # x_buf after the BA
    fb = b.factor().export()
    assert ref.value("factor_size", lambda: len(a.factor().export()["sum10"])) == len(fb["sum10"]) > 20
    pa, pb = a and a.planes(), b.planes()
    ka, kb = pa and np.lexsort(np.round(pa["voxel_center"], 9).T), np.lexsort(np.round(pb["voxel_center"], 9).T)
    P = ref.rows("planes", lambda: _plane_rows(pa, ka, "cov_trace"))
    assert P.n == len(pb["N"]) > 20
    assert ref.digest("plane_N", lambda: pa["N"][ka]) == digest(pb["N"][kb])
    Pb = _plane_rows(pb, kb, "cov_trace")[P.idx]
    Pa = P.rows
    assert np.max(np.abs(Pa[:, :3] - Pb[:, :3])) < 1e-9
    assert np.max(np.abs(Pa[:, 42] - Pb[:, 42]) / Pb[:, 42]) < 1e-10    # the Bf_var accumulation with full variances
    Vb = _flip_by_normal(Pa, Pb)
    assert np.max(np.abs(Pa[:, 6:42].reshape(-1, 6, 6) - Vb) / np.max(np.abs(Vb), axis=(1, 2), keepdims=True)) < 1e-5
    pose = synth.perturb_pose(synth.true_pose(L, nscan), 78, 1e-3, 5e-3)
    pv = _pv_records(synth.gen_scan(L, nscan, 3000, synth.true_pose(L, nscan), seed=0x5EED0000 + 33), 99)
    oa_ = a and a.odom_accumulate(pv, pose, np.eye(3) * 1e-6, np.eye(3) * 1e-5)
    ob_ = b.odom_accumulate(pv, pose, np.eye(3) * 1e-6, np.eye(3) * 1e-5)
    o = ref.value("odom", lambda: {k: oa_[k] for k in ("n", "HTH", "HTz")})
    assert o["n"] == ob_["n"] > 300 and ref.digest("odom_flags", lambda: oa_["flags"]) == digest(ob_["flags"])
    assert relinf(o["HTH"], ob_["HTH"]) < 1e-8 and relinf(o["HTz"], ob_["HTz"]) < 1e-8


def test_var_init_and_pvec_update_against_the_reference_functions(ref):
    """calcBodyVar / var_init / pvec_update (voxelslam.hpp:163-214, cut out of voxelslam.hpp at build time): the restatement vs the reference's code,
    incl. a point with z == 0 (the reference moves it to z = 1e-4) and points on the axes' neighbourhood."""
    ra = ref.ra
    rng = np.random.default_rng(5)
    n = 4000
    pts = np.zeros((n, 12), dtype=np.float32)                       # PointType stride (12 floats)
    pts[:, :3] = rng.uniform(-40, 40, (n, 3)).astype(np.float32)
    pts[0, :3] = (3.0, -2.0, 0.0)                                  # z == 0 trap (voxelslam.hpp:165)
    pts[1, :3] = (0.01, 0.02, 35.0)
    pts[2, :3] = (25.0, -25.0, 1e-3)
    ext_R = oa.so3_exp(np.array([0.02, -0.01, 0.03])); ext_p = np.array([0.05, -0.02, 0.1])
    a = oa.var_init(pts, ext_R, ext_p, 0.02, 0.05)
    b = ra and ra.var_init(pts, ext_R, ext_p, 0.02, 0.05)
    assert ref.digest("var_init_pnt", lambda: b[:, :3]) == digest(a[:, :3])
    B = ref.rows("var_init_var", lambda: b[:, 3:])
    assert B.n == n and np.max(np.abs(a[B.idx, 3:] - B.rows) / (np.max(np.abs(B.rows), axis=1, keepdims=True))) < 1e-12
    assert abs(a[0, 2] - (ext_R @ np.array([3.0, -2.0, 1e-4]) + ext_p)[2]) < 1e-15
    pose = np.concatenate([oa.so3_exp(np.array([0.3, 0.1, -0.2])).ravel(), [5.0, -3.0, 1.0]])
    A = rng.standard_normal((3, 3)) * 1e-3; rot_var = A @ A.T
    B = rng.standard_normal((3, 3)) * 1e-2; tsl_var = B @ B.T
    pa, wa = oa.pvec_update(a, pose, rot_var, tsl_var)
    pb, wb = ra and ra.pvec_update(a, pose, rot_var, tsl_var) or (None, None)
    assert np.array_equal(pa[:, :3], a[:, :3])                      # pnt stays in the body frame
    Wb = ref.rows("pvec_update_pwld", lambda: wb)
    assert Wb.n == n and np.max(np.abs(wa[Wb.idx] - Wb.rows)) < 1e-12
    Pb = ref.rows("pvec_update_var", lambda: pb[:, 3:])
    assert Pb.n == n and np.max(np.abs(pa[Pb.idx, 3:] - Pb.rows) / np.max(np.abs(Pb.rows), axis=1, keepdims=True)) < 1e-12


@pytest.mark.parametrize("max_iter", [1, 4])
def test_hba_add_edge_against_the_reference_member_function(max_iter, ref):
    """The reference's own HBA_add_edge (voxelslam.cpp:2319-2482, cut out of the ROS node class at build time): coarse -> fine outer loop over OctreeGBA map
    builds and Lidar_BA_Optimizer solves, the PGO edges of the final Hessian and the merged + down-sampled submap — against the oracle's hba_window /
    hba_edges / submap_merge chain that the GPU tests (vxs_hba_window, vxs_hba_edges, vxs_submap_merge, vxs_hba_bottom_batch, vxs_hba_pass) compare with.
    The reference optimises a private copy of the poses, so they are pinned through the edges' relative poses and the merged cloud."""
    W = 8
    tr, est = scenes.poses_true_est(W, 8.0, 43, rot_sigma=3e-3, pos_sigma=2e-2)
    xyz, off = scenes.make_points(W, 4000, 8.0, 43, tr, dtype=np.float32)
    coarse = vx.MapParams.make(voxel_size=2.0, min_eigen_value=0.1, max_layer=2)
    fine = vx.MapParams.make(voxel_size=1.0, min_eigen_value=0.0025, max_layer=2)
    r = ref.ra and ref.ra.hba_add_edge(coarse, fine, xyz, off, est, max_iter, thread_num=2)
    a = ref.value("edges", lambda: {k: r[k] for k in ("n", "ij", "v6", "rot", "tra")})
    w = oa.hba_window(coarse, fine, xyz, off, est, max_iter, thread_num=2)
    assert w["status"] == 0 and w["outer_iters"] == max_iter
    e = oa.hba_edges(w["hess"], W, w["poses"])
    assert a["n"] == e["n"] == W * (W - 1) // 2 and np.array_equal(a["ij"], e["ij"])      # lexicographic (i, j), voxelslam.cpp:2405-2406
    assert np.max(np.abs(a["v6"] - e["v6"]) / np.abs(e["v6"])) < 1e-10
    assert np.max(np.abs(a["rot"] - e["rot"])) < 1e-12 and np.max(np.abs(a["tra"] - e["tra"])) < 1e-12
    assert np.max(np.abs(w["poses"] - est)) > 1e-4                                       # the solve moved the poses: the edges above are not the input's
    m = oa.submap_merge(xyz, off, w["poses"], fine.voxel_size / 8)
    assert ref.value("submap_n", lambda: len(r["submap"])) == len(m["xyz"]) > 1000
    kb = np.lexsort(m["xyz"].T)
    assert ref.digest("submap", lambda: r["submap"][np.lexsort(r["submap"].T)].view(np.uint32)) == digest(m["xyz"][kb].view(np.uint32))  # float running means of the same cells, bit-exact


def _hat(v):
    return np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])


def _so3_log(R):                      # tools.hpp:86-91
    tr_ = np.trace(R)
    th = 0.0 if tr_ > 3.0 - 1e-6 else np.arccos(0.5 * (tr_ - 1))
    K = np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]])
    return 0.5 * K if abs(th) < 0.001 else 0.5 * th / np.sin(th) * K


def _ekf_update_numpy(accum, pv, st, cov, num_max_iter=4):
    """lio_state_estimation (voxelslam.cpp:856-954) with its association + accumulation loop (:876-918) replaced by `accum`: a FULL match of every point in
    every iteration — what vxs_odom_accumulate / vxs_map_odom_accumulate do — instead of the reference's per-point leaf cache (octos[i])."""
    x_prop, x, cov = st.copy(), st.copy(), cov.copy()
    G, H15, I15 = np.zeros((15, 15)), np.zeros((15, 15)), np.eye(15)
    rematch = 0
    cov_inv = np.linalg.inv(cov)
    for it in range(num_max_iter):
        o = accum(pv, x[:12], cov[:3, :3], cov[3:6, 3:6])
        H15[:6, :6] = o["HTH"]
        K1 = np.linalg.inv(H15 + cov_inv)
        G[:, :6] = K1[:, :6] @ o["HTH"]
        vec = np.zeros(15)                                                          # x_prop - x_curr, IMUST::operator- (tools.hpp:164-173)
        vec[:3] = _so3_log(x[:9].reshape(3, 3).T @ x_prop[:9].reshape(3, 3)); vec[3:] = x_prop[9:21] - x[9:21]
        sol = K1[:, :6] @ o["HTz"] + vec - G[:, :6] @ vec[:6]
        x = x.copy(); x[:9] = (x[:9].reshape(3, 3) @ oa.so3_exp(sol[:3])).ravel(); x[9:21] += sol[3:]   # IMUST::operator+= (tools.hpp:154-162)
        conv = np.linalg.norm(sol[:3]) * 57.3 < 0.01 and np.linalg.norm(sol[3:6]) * 100 < 0.015
        if conv or (rematch == 0 and it == num_max_iter - 2):
            rematch += 1
        if rematch >= 2 or it == num_max_iter - 1:
            cov = (I15 - G) @ cov
            break
    return bool(np.linalg.eigvalsh(o["nnt"])[0] >= 14), x, cov, o["n"]


@pytest.mark.parametrize("sigma", [0.01, 0.12])
def test_lio_state_estimation_against_the_reference_member_function(sigma, ref):
    """The reference's whole odometry update (lio_state_estimation, voxelslam.cpp:856-954, cut out of the node class at build time: up to 4 EKF iterations, each
    re-associating the scan through its per-point leaf cache) against the oracle's accumulation with a full match per iteration + the 15x15 EKF algebra in numpy.
    Equal to rounding -> the leaf cache is a pure shortcut and the CUDA path (no cache, full match per call) reproduces the reference's update; sigma = 0.12
    leaves ~30 % of the points unmatched (3-sigma gates), which is where a cached leaf and a fresh descent could disagree."""
    W, L = 4, 6.0
    tr, est = scenes.poses_true_est(W, L, 5)
    pts, off = scenes.make_points(W, 6000, L, 5, tr)
    mp = vx.MapParams.make(voxel_size=1.0, max_layer=2)
    a, b = ref.ra and ref.ra.LocalMap(mp, pts, off, tr, 1e-4, mgsize=1), oa.LocalMap(mp, pts, off, tr, 1e-4, mgsize=1)
    scan = synth.gen_scan(L, W - 1, 4000, tr[W - 1], seed=0x5EED0000 + 5, sigma=sigma)
    pv = np.zeros((scan.shape[0], 12)); pv[:, :3] = scan; pv[:, [3, 7, 11]] = 1e-4
    for seed, rs, ps in ((77, 1e-3, 5e-3), (79, 2e-2, 8e-2)):
        st = np.zeros(24); st[:12] = synth.perturb_pose(tr[W - 1], seed, rs, ps); st[12:15] = (0.3, -0.1, 0.05); st[21:24] = (0, 0, -9.8)
        cov = np.diag([1e-4] * 3 + [1e-3] * 3 + [1e-2] * 3 + [1e-6] * 6)
        r = ref.value(f"lio_{seed}", lambda: dict(zip(("ok", "state", "cov"), a.lio_state_estimation(pv, st, cov))))
        ok_r, st_r, cov_r = r["ok"], r["state"], r["cov"]
        ok_o, st_o, cov_o, nm = _ekf_update_numpy(lambda p_, x_, rv, tv: b.odom_accumulate(p_, x_, rv, tv, passes=1), pv, st, cov)
        assert ok_r == ok_o and (nm == 4000 if sigma < 0.05 else 2000 < nm < 3500)
        assert np.max(np.abs(st_r[:21] - st_o[:21])) < 1e-12 and np.max(np.abs(cov_r - cov_o)) / np.max(np.abs(cov_o)) < 1e-12
        assert np.max(np.abs(st_r[:12] - st[:12])) > 3e-3                                   # the update moved the state ...
        if sigma < 0.05 or ps > 0.05:                                                          # (a 5 mm start error is below what a 12 cm noise scan resolves)
            assert np.max(np.abs(st_r[9:12] - tr[W - 1][9:12])) < np.max(np.abs(st[9:12] - tr[W - 1][9:12]))   # ... towards the truth
