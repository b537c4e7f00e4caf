"""Pins the oracle (and the product's host-side file logic) against the reference's OWN code.

oracle/_ref/libltremovert_ref.so holds ltremovert/src/{utility,RosParamServer,Session,Removerter}.cpp compiled unmodified
from the reference's sources against stand-in third-party headers (oracle/ref_shim/include/ltr_shim_core.h).  Every comparison is
bit-exact.  What this pins: all first-party logic (projection, pixel indexing, min selection, discrepancy thresholds, index
set arithmetic, kNN threshold test, schedule / run() order, keyframe parsing, pose reading).  What it does not: the
third-party algorithms, whose stand-ins call the oracle's restatements (PCL transform / octree centroid / FLANN kNN / Eigen
inverse).

CPU only.  The reference's answers are replayed from tests/golden/ref_pin.json.gz (oracle/ref_golden.py), recorded from
oracle/_ref where the reference's sources are available:  LTR_RECORD_REFERENCE=1 python -m pytest -p no:xdist tests/test_ref_pin.py
"""
import os

import numpy as np
import pytest

import oracle
from oracle.ref_golden import RecordedRef, bits_equal, values_equal
from lt_mapper_b200 import removert

ref = RecordedRef(os.path.join(os.path.dirname(__file__), "golden", "ref_pin.json.gz"))

EXT = np.array([[np.cos(0.3), -np.sin(0.3), 0, 0.5], [np.sin(0.3), np.cos(0.3), 0, -0.2], [0, 0, 1, 1.1], [0, 0, 0, 1.0]])


@pytest.fixture(scope="module", autouse=True)
def _save_recording(request):
    yield
    ref.rec.save(request.session.testsfailed == 0)


@pytest.fixture(autouse=True)
def _reference_calls(request):
    with ref.rec.test(request.node.name):
        yield


def write_pcd(path, a):
    a = np.ascontiguousarray(a, np.float32)
    with open(path, "wb") as f:
        f.write((f"# .PCD v0.7 - Point Cloud Data file format\nVERSION 0.7\nFIELDS x y z intensity\nSIZE 4 4 4 4\nTYPE F F F F\n"
                 f"COUNT 1 1 1 1\nWIDTH {len(a)}\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS {len(a)}\nDATA binary\n").encode())
        f.write(a.tobytes())


def write_session(d, s, extra_poses=()):
    os.makedirs(os.path.join(d, "scans"), exist_ok=True)
    for k in range(s.K):
        write_pcd(os.path.join(d, "scans", f"{k:06d}.pcd"), s.scan(k))
    with open(os.path.join(d, "poses.txt"), "w") as f:
        for P in list(s.poses) + list(extra_poses):
            f.write(" ".join(repr(float(v)) for v in P[:3].ravel()) + "\n")


def base_params(root, l2b=np.eye(4), **kw):
    p = dict(central_sess_scan_dir=f"{root}/central/scans", central_sess_pose_path=f"{root}/central/poses.txt",
             query_sess_scan_dir=f"{root}/query/scans", query_sess_pose_path=f"{root}/query/poses.txt",
             save_pcd_directory=f"{root}/out/", sequence_vfov=50.0, sequence_hfov=360.0,
             ExtrinsicLiDARtoPoseBase=np.asarray(l2b, np.float64).ravel().tolist(), downsample_voxel_size=0.05,
             num_nn_points_within=2, dist_nn_points_within=0.01, start_idx=0, end_idx=1000, keyframe_gap=1,
             remove_resolution_list=[2.5, 2.0, 1.5], revert_resolution_list=[1.0], num_omp_cores=4, saveMapPCD=True)
    p.update(kw)
    return p


@pytest.fixture(scope="module")
def session_files(small_pair, tmp_path_factory):
    root = str(tmp_path_factory.mktemp("refpin"))
    write_session(root + "/central", small_pair[0])
    write_session(root + "/query", small_pair[1])
    return root


@pytest.fixture(scope="module")
def scratch(tmp_path_factory):
    """save_pcd_directory for runs that save nothing (the node's constructor still creates its output tree, Removerter.cpp:26-49)."""
    return str(tmp_path_factory.mktemp("refscratch"))


# ------------------------------------------------------------------------------------------------ scalar level
def _probe_points(rng):
    pts = [rng.normal(0, s, (20000, 3)) for s in (0.01, 1.0, 30.0, 300.0)]
    axes = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1], [0, 0, 0], [-1, 1e-30, 0], [-1, -1e-30, 0],
                     [1e-20, 1e-20, 1e-20], [1e18, -1e18, 1e18], [-3, 0.0, 2], [-3, -0.0, 2]], np.float64)
    return np.concatenate(pts + [axes]).astype(np.float32)


def test_cart2sph_and_rad2deg_match_the_reference():
    p = _probe_points(np.random.default_rng(1))
    got = ref.cart2sph(p)
    x, y, z = p[:, 0], p[:, 1], p[:, 2]
    exp = np.stack([oracle.atan2f(y, x), oracle.atan2f(z, np.sqrt(x * x + y * y)), np.sqrt(x * x + y * y + z * z)], 1)
    assert bits_equal(got, exp)
    assert bits_equal(exp[:, 2], oracle.pixel_index(p, 125, 900)[2])
    a = np.concatenate([exp[:, 0], exp[:, 1]])
    assert bits_equal(ref.rad2deg(a), (a.astype(np.float64) * 180.0 / np.pi).astype(np.float32))


@pytest.mark.parametrize("alpha", [0.5, 0.95, 1.0, 1.425, 1.5, 2.0, 2.375, 2.5, 3.0])
def test_rimg_size_matches_the_reference(alpha):
    for vfov, hfov in ((50.0, 360.0), (40.0, 360.0), (33.2, 180.0)):
        assert ref.reset_rimg_size(alpha, vfov, hfov) == oracle.reset_rimg_size(alpha, vfov, hfov)


def test_range_images_match_the_reference(small_pair, scratch):
    c = small_pair[0]
    R = ref.Removerter(base_params(scratch), write_files=False)
    scan = c.scan(2)
    both = np.concatenate([scan, scan[::-1], _probe_points(np.random.default_rng(2))[:, [0, 1, 2, 0]]])   # duplicates -> range ties
    for alpha in (0.5, 1.0, 2.5, 3.0):
        rows, cols = oracle.reset_rimg_size(alpha)
        for cloud in (scan, both):
            er, ei = oracle.map2rimg(cloud, rows, cols)
            gr, gi = ref.map2rimg(cloud, rows, cols)
            assert bits_equal(gr, er) and bits_equal(gi, ei)
            assert bits_equal(R.scan2rimg(cloud, rows, cols), oracle.scan2rimg(cloud, rows, cols))
    R.close()


def test_global_to_local_and_projected_parse_match_the_reference(small_pair, small_maps, scratch):
    c = small_pair[0]
    m = small_maps[0]
    for order, l2b in ((0, np.eye(4)), (1, EXT)):
        R = ref.Removerter(base_params(scratch, l2b), transform_order=order, write_files=False)
        _, b2l = R.extrinsics()
        assert bits_equal(b2l, oracle.inverse4x4(l2b))
        for k in (0, 3):
            ip = oracle.inverse4x4(c.poses[k])
            assert bits_equal(ref.inverse4x4(c.poses[k]), ip)
            loc = ref.transform_global_to_local(m, ip, b2l)
            assert bits_equal(loc, oracle.transform(oracle.transform(m, ip, order), b2l, order))
            rows, cols = oracle.reset_rimg_size(3.0)
            exp, _ = oracle.parse_projected(m, ip, 3.0, lidar2base=l2b, order=order)
            assert bits_equal(ref.parse_projected(loc, rows, cols), exp)
        R.close()


def test_index_set_arithmetic_matches_the_reference(scratch):
    # linspace<int>(0, N, N) (utility.h:158-167): integer step N / (N - 1) == 1 for N >= 3 -> 0 .. N-1
    for n in (3, 4, 17, 1000):
        assert values_equal(ref.linspace_int(0, n, n), np.arange(n))
    assert values_equal(ref.linspace_int(0, 2, 2), [0, 2])      # the N == 2 quirk the oracle / product document (index 2 is out of range)
    R = ref.Removerter(base_params(scratch), write_files=False)
    rng = np.random.default_rng(3)
    for n in (3, 50, 5000):
        dyn = np.unique(rng.integers(0, n, n // 3)).astype(np.int32)
        assert values_equal(R.static_idx(dyn, n), np.setdiff1d(np.arange(n), dyn))
    R.close()


# ------------------------------------------------------------------------------------------------ pass level
@pytest.mark.parametrize("order,l2b", [(0, np.eye(4)), (1, EXT)])
def test_remove_nd_pd_passes_match_the_reference(small_pair, small_maps, scratch, order, l2b):
    c, q = small_pair
    R = ref.Removerter(base_params(scratch, l2b), transform_order=order, write_files=False)
    R.load_session_mem(0, c.xyzi, c.offsets, c.poses)
    R.load_session_mem(1, q.xyzi, q.offsets, q.poses)
    inv = [np.stack([ref.inverse4x4(p) for p in s.poses]) for s in (c, q)]
    m = small_maps[0]
    # HD (Removerter.cpp:542-593): target map vs the source session's raw keyframe scans, threshold 0.1
    for alpha in (2.5, 1.0):
        rows, cols = oracle.reset_rimg_size(alpha)
        R.set_cloud("map_global_curr_", m, 0)
        got = R.dynamic_idx(0, 0, 0, rows, cols, len(m))
        exp = oracle.remove_pass(m, c.xyzi, c.offsets, inv[0], oracle.MODE_HD, alpha, 0.1, lidar2base=l2b, order=order)
        assert values_equal(got, np.flatnonzero(exp))
        assert len(got) > 100
    # ND (:485-540) and PD (:429-482) read the source session's keyframe_scans_static_projected_
    R.set_scans("keyframe_scans_static_projected_", q.xyzi, q.offsets, 1)
    rows, cols = oracle.reset_rimg_size(2.5)
    R.set_cloud("map_global_nd_", m, 0)
    got = R.dynamic_idx(1, 0, 1, rows, cols, len(m))
    exp = oracle.remove_pass(m, q.xyzi, q.offsets, inv[1], oracle.MODE_ND, 2.5, 0.1, lidar2base=l2b, order=order)
    assert values_equal(got, np.flatnonzero(exp)) and len(got) > 10
    R.set_cloud("map_global_pd_", m, 0)
    got = R.dynamic_idx(2, 0, 1, rows, cols, len(m))
    exp = oracle.remove_pass(m, q.xyzi, q.offsets, inv[1], oracle.MODE_PD, 2.5, 0.1, lidar2base=l2b, order=order)
    assert values_equal(got, np.flatnonzero(exp)) and len(got) > 10
    R.close()


# ------------------------------------------------------------------------------------------------ pipeline level
CLOUDS_AFTER = {
    "precleaningKeyframes": ([], ["keyframe_scans_"]),
    "makeGlobalMap": (["map_global_orig_", "map_global_curr_"], []),
    "removeHighDynamicPoints": (["map_global_curr_", "map_global_curr_static_", "map_global_curr_dynamic_"], ["keyframe_scans_dynamic_"]),
    "parseStaticScansViaProjection": ([], ["keyframe_scans_static_projected_"]),
    "detectLowDynamicPoints": (["map_global_nd_", "map_global_nd_strong_", "map_global_nd_weak_", "map_global_pd_", "map_global_pd_orig_",
                                "map_global_pd_strong_", "map_global_pd_weak_"], ["scans_knn_coexist_", "scans_knn_diff_"]),
    "updateCurrentMap": (["map_global_updated_", "map_global_updated_strong_"], []),
    "parseUpdatedStaticScansViaProjection": ([], ["keyframe_scans_updated_", "keyframe_scans_updated_strong_"]),
    "parseLDScansViaProjection": ([], ["keyframe_scans_pd_", "keyframe_scans_strong_pd_", "keyframe_scans_strong_nd_", "keyframe_scans_weak_nd_"]),
    "updateScansScanwise": ([], ["keyframe_scans_updated_"]),
}
SAVED = ["OriginalNoisyCentralMapGlobal", "OriginalNoisyQueryMapGlobal", "central_sess_high_dyn", "query_sess_high_dyn", "union_map_queryside",
         "union_map_centralside", "pd_map", "nd_map", "strong_nd_map", "weak_nd_map", "strong_pd_map", "weak_pd_map", "updated_map", "updated_map_strong"]


def _load_oracle_from_ref(R, O, scans):
    """scans[s]: the keyframe scans the reference loaded for session s (checked equal to R.scans("keyframe_scans_", s) by the caller)."""
    for s in (0, 1):
        sc = scans[s]
        P, IP = R.keyframe_poses(s)
        off = np.concatenate([[0], np.cumsum([len(a) for a in sc])]).astype(np.int64)
        O.load_session(s, np.concatenate(sc), off, P, IP)


@pytest.mark.parametrize("order,l2b,knn,thr", [(0, np.eye(4), 2, 0.01), (1, EXT, 1, 0.04), (0, EXT, 3, 0.1)])
def test_run_matches_the_reference_stage_by_stage(session_files, small_pair, order, l2b, knn, thr):
    root = session_files
    R = ref.Removerter(base_params(root, l2b, num_nn_points_within=knn, dist_nn_points_within=thr), transform_order=order)
    for st in ("loadSessionInfo", "parseKeyframes", "loadKeyframes"):
        R.stage(st)
    assert R.num_keyframes(0) == small_pair[0].K and R.num_keyframes(1) == small_pair[1].K
    # file reading + pcl::VoxelGrid of Session::loadKeyframes against the product's host helpers
    loaded = []
    for s in (0, 1):
        P, IP = R.keyframe_poses(s)
        assert bits_equal(P, removert.read_poses(f"{root}/{'central' if s == 0 else 'query'}/poses.txt"))
        got = R.scans("keyframe_scans_", s)
        loaded.append([removert.voxel_grid(small_pair[s].scan(k), 0.05)[0] for k in range(small_pair[s].K)])
        assert len(got) == len(loaded[s]) and all(bits_equal(a, b) for a, b in zip(got, loaded[s]))
    O = oracle.Removerter(num_knn=knn, knn_thr=thr, voxel=0.05, order=order, lidar2base=l2b, threads=4)
    _load_oracle_from_ref(R, O, loaded)
    for st, (clouds, scansets) in CLOUDS_AFTER.items():
        R.stage(st)
        O.stage(st)
        for s in (0, 1):
            for name in clouds:
                assert bits_equal(R.cloud(name, s), O.cloud(name, s)), (st, name, s)
            for name in scansets:
                got = R.scans(name, s)
                if s == 1 and not got:
                    continue                                  # Step 3 only touches the central session
                exp = O.clouds(name, s)
                assert len(got) == len(exp) and all(bits_equal(a, b) for a, b in zip(got, exp)), (st, name, s)
    R.stage("saveAllTypeOfScans")
    saved = {os.path.basename(p)[:-4]: a for p, a in R.saved() if os.path.dirname(p) == os.path.normpath(root + "/out")}
    assert sorted(saved) == sorted(SAVED)
    for name in SAVED:
        assert bits_equal(saved[name], O.cloud("saved:" + name)), name
    # the per-keyframe scan files of Step 3 (Removerter.cpp:1637-1650) and what lands on disk
    names = R.keyframe_names(0)
    for sub, member in (("scans_updated", "keyframe_scans_updated_"), ("scans_updated_strong", "keyframe_scans_updated_strong_"),
                        ("scans_pd", "keyframe_scans_pd_"), ("scans_pd_strong", "keyframe_scans_strong_pd_"), ("scans_nd_strong", "keyframe_scans_strong_nd_")):
        exp = O.clouds(member, 0)
        for k, nm in enumerate(names):
            written = ref.capture("file written", (sub, nm), lambda: removert.read_pcd(f"{root}/out/{sub}/{nm}"))
            assert bits_equal(written, exp[k]), (sub, nm)
    R.close()


def test_multi_resolution_schedules_match_the_reference(small_pair, scratch):
    """selfRemovert (Removerter.cpp:1378-1393) and the BASELINE remove x3 + revert schedule, driven op by op on the reference."""
    c = small_pair[0]
    R = ref.Removerter(base_params(scratch, remove_resolution_list=[2.5, 1.5]), write_files=False)
    R.load_session_mem(0, c.xyzi, c.offsets, c.poses)
    R.load_session_mem(1, c.xyzi[:0], np.zeros(1, np.int64), c.poses[:0])
    R.stage("precleaningKeyframes"); R.stage("makeGlobalMap")
    m0 = R.cloud("map_global_curr_", 0)
    sched = removert.selfremovert_schedule([2.5, 1.5])
    O = oracle.Removerter(schedule=sched, threads=4, do_high_dyn_knn=False)
    O.load_session(0, c.xyzi, c.offsets, c.poses, np.stack([ref.inverse4x4(p) for p in c.poses]))
    O.load_session(1, c.xyzi[:0], np.zeros(1, np.int64), c.poses[:0])
    O.stage("precleaningKeyframes"); O.stage("makeGlobalMap")
    assert bits_equal(m0, O.cloud("map_global_curr_", 0))
    R.self_removert(0, 1)
    O.stage("removeHighDynamicPoints")
    for name in ("map_global_curr_", "map_global_curr_static_", "map_global_curr_dynamic_"):
        assert bits_equal(R.cloud(name, 0), O.cloud(name, 0)), name
    # the schedule bench.py runs: removeOnce at 2.5, 2.0, 1.5, then one revert at 1.0
    none = np.zeros((0, 4), np.float32)
    R.set_cloud("map_global_curr_", m0, 0); R.set_cloud("map_global_curr_static_", none, 0); R.set_cloud("map_global_curr_dynamic_", none, 0)
    for res in (2.5, 2.0, 1.5):
        R.op("removeOnce", 0, 0, res)
    R.op("resetAsDynamic", 0); R.op("revertOnce", 0, 0, 1.0); R.op("resetAsStatic", 0)
    O2 = oracle.Removerter(schedule=[(0, 2.5), (0, 2.0), (0, 1.5), (1, 1.0)], threads=4, do_high_dyn_knn=False)
    O2.load_session(0, c.xyzi, c.offsets, c.poses, np.stack([ref.inverse4x4(p) for p in c.poses]))
    O2.load_session(1, c.xyzi[:0], np.zeros(1, np.int64), c.poses[:0])
    O2.stage("precleaningKeyframes"); O2.stage("makeGlobalMap"); O2.stage("removeHighDynamicPoints")
    for name in ("map_global_curr_", "map_global_curr_static_", "map_global_curr_dynamic_"):
        assert bits_equal(R.cloud(name, 0), O2.cloud(name, 0)), name
    R.close()


# ------------------------------------------------------------------------------------------------ host logic
@pytest.mark.parametrize("start,end,gap", [(0, 1000, 1), (0, 1000, 2), (1, 4, 1), (2, 3, 1), (3, 5, 2), (5, 5, 1)])
def test_keyframe_parsing_matches_the_reference(session_files, small_pair, start, end, gap):
    root = session_files
    R = ref.Removerter(base_params(root, start_idx=start, end_idx=end, keyframe_gap=gap), write_files=False)
    R.stage("loadSessionInfo"); R.stage("parseKeyframes")
    n = small_pair[0].K
    assert R.num_scans(0) == n
    exp_c = list(removert.parse_keyframes(n, start, end, gap))
    assert R.keyframe_names(0) == [f"{k:06d}.pcd" for k in exp_c]
    central_kf_poses = R.keyframe_poses(0)[0]
    q_poses = removert.read_poses(f"{root}/query/poses.txt")
    exp_q = list(removert.parse_keyframes_in_roi(q_poses, central_kf_poses, gap))
    assert R.keyframe_names(1) == [f"{k:06d}.pcd" for k in exp_q]
    R.close()


def test_schedule_driven_step1_matches_the_reference(small_pair, scratch):
    """ref_high_dyn_with_schedule (what bench.py --impl reference times) == the oracle's scheduled Step 1, both sessions."""
    sched = [(0, 2.5), (0, 2.0), (0, 1.5), (1, 1.0)]
    R = ref.Removerter(base_params(scratch, num_nn_points_within=1, dist_nn_points_within=0.04), write_files=False)
    O = oracle.Removerter(schedule=sched, num_knn=1, knn_thr=0.04, threads=4)
    for s, d in enumerate(small_pair):
        R.load_session_mem(s, d.xyzi, d.offsets, d.poses)
        O.load_session(s, d.xyzi, d.offsets, d.poses, np.stack([ref.inverse4x4(p) for p in d.poses]))
    for st in ("precleaningKeyframes", "makeGlobalMap"):
        R.stage(st); O.stage(st)
    R.high_dyn_with_schedule(sched)
    O.stage("removeHighDynamicPoints")
    for st in ("parseStaticScansViaProjection", "detectLowDynamicPoints"):
        R.stage(st); O.stage(st)
    for s in (0, 1):
        for name in ("map_global_curr_", "map_global_curr_static_", "map_global_curr_dynamic_", "map_global_nd_strong_", "map_global_nd_weak_",
                     "map_global_pd_strong_", "map_global_pd_weak_"):
            assert bits_equal(R.cloud(name, s), O.cloud(name, s)), (name, s)
        for name in ("keyframe_scans_dynamic_", "keyframe_scans_static_projected_", "scans_knn_diff_"):
            got, exp = R.scans(name, s), O.clouds(name, s)
            assert len(got) == len(exp) and all(bits_equal(a, b) for a, b in zip(got, exp)), (name, s)
    R.close()


@pytest.mark.parametrize("vfov,hfov", [(40.0, 360.0), (33.2, 180.0), (90.0, 360.0), (50.0, 359.0)])
def test_non_default_fov_matches_the_reference(small_pair, small_maps, scratch, vfov, hfov):
    """sequence_vfov / sequence_hfov other than the yaml's 50 x 360: image size, pixel clamping and the HD index set."""
    c = small_pair[0]
    m = small_maps[0]
    R = ref.Removerter(base_params(scratch, sequence_vfov=vfov, sequence_hfov=hfov), write_files=False)
    R.load_session_mem(0, c.xyzi, c.offsets, c.poses)
    inv = np.stack([ref.inverse4x4(p) for p in c.poses])
    for alpha in (2.5, 0.7):
        rows, cols = oracle.reset_rimg_size(alpha, vfov, hfov)
        assert (rows, cols) == ref.reset_rimg_size(alpha, vfov, hfov)
        R.set_cloud("map_global_curr_", m, 0)
        got = R.dynamic_idx(0, 0, 0, rows, cols, len(m))
        exp = oracle.remove_pass(m, c.xyzi, c.offsets, inv, oracle.MODE_HD, alpha, 0.1, vfov=vfov, hfov=hfov)
        assert values_equal(got, np.flatnonzero(exp)) and len(got) > 100
    R.close()


@pytest.mark.parametrize("seed,beams,az", [(99, 16, 1200), (2024, 48, 600)])
def test_full_run_on_other_scenes_matches_the_reference(scratch, seed, beams, az):
    """Removerter::run() end to end (in-memory load, Steps 0-3) on differently seeded / shaped synthetic scenes."""
    import synth
    pair = synth.make_pair(5, beams=beams, az_steps=az, seed=seed)
    R = ref.Removerter(base_params(scratch), write_files=False)
    O = oracle.Removerter(num_knn=2, knn_thr=0.01, threads=4)
    for s, d in enumerate(pair):
        R.load_session_mem(s, d.xyzi, d.offsets, d.poses)
        O.load_session(s, d.xyzi, d.offsets, d.poses, np.stack([ref.inverse4x4(p) for p in d.poses]))
    for st in CLOUDS_AFTER:
        R.stage(st); O.stage(st)
    for name in ("map_global_curr_static_", "map_global_curr_dynamic_", "map_global_nd_strong_", "map_global_nd_weak_", "map_global_pd_strong_",
                 "map_global_pd_weak_", "map_global_updated_", "map_global_updated_strong_"):
        for s in (0, 1):
            assert bits_equal(R.cloud(name, s), O.cloud(name, s)), (name, s)
    for name in ("keyframe_scans_updated_", "keyframe_scans_pd_", "keyframe_scans_strong_nd_"):
        got, exp = R.scans(name, 0), O.clouds(name, 0)
        assert len(got) == len(exp) == 5 and all(bits_equal(a, b) for a, b in zip(got, exp)), name
    assert len(R.cloud("map_global_curr_dynamic_", 0)) > 0
    R.close()


def test_property_random_clouds_match_the_reference():
    """Property test (hypothesis): arbitrary finite float32 clouds -- including zeros, signed zeros, denormals, huge and tiny magnitudes,
    duplicated points -- give bit-identical cart2sph values and range / index images in the compiled reference and in the oracle."""
    from hypothesis import given, settings, strategies as st, HealthCheck
    f32 = st.floats(width=32, allow_nan=False, allow_infinity=False, min_value=-1e6, max_value=1e6)
    special = st.sampled_from([0.0, -0.0, 1e-38, -1e-38, 1e-45, 1.0, -1.0, 100.0, -100.0, 1e6, 3.4e5, 2.5, 0.5])
    coord = st.one_of(f32, special)
    pts = st.lists(st.tuples(coord, coord, coord), min_size=1, max_size=200)

    def check(p, alpha, dup):
        a = np.array(p, np.float32).reshape(-1, 3)
        if dup:
            a = np.concatenate([a, a[::-1]])
        cloud = np.concatenate([a, np.zeros((len(a), 1), np.float32)], 1)
        got = ref.cart2sph(a)
        x, y, z = a[:, 0], a[:, 1], a[:, 2]
        with np.errstate(all="ignore"):
            assert bits_equal(got, np.stack([oracle.atan2f(y, x), oracle.atan2f(z, np.sqrt(x * x + y * y)), np.sqrt(x * x + y * y + z * z)], 1))
        rows, cols = oracle.reset_rimg_size(alpha)
        er, ei = oracle.map2rimg(cloud, rows, cols)
        gr, gi = ref.map2rimg(cloud, rows, cols)
        assert bits_equal(gr, er) and bits_equal(gi, ei)
        # parseProjectedPoints (utility.cpp:74-89): row-major emission, the point with index 0 is never emitted
        cloud[:, 3] = np.arange(len(cloud), dtype=np.float32)
        exp, idx = oracle.parse_projected(cloud, np.eye(4), alpha)
        loc = ref.transform_global_to_local(cloud, np.eye(4), np.eye(4))   # as Session::parseScansViaProjection does (turns -0.0 into +0.0)
        assert bits_equal(ref.parse_projected(loc, rows, cols), exp) and 0 not in idx
    ref.rec.examples(check, lambda f: settings(max_examples=60, deadline=None, suppress_health_check=list(HealthCheck))(
        given(pts, st.sampled_from([0.1, 0.4, 2.5, 3.0]), st.booleans())(f)))


def test_property_random_passes_match_the_reference(scratch):
    """Property test: small random maps and scans (not geometrically consistent, coarse images so that pixels collide, duplicated points so that
    ranges tie) through the three pass variants of the compiled reference and of the oracle: identical dynamic index sets."""
    from hypothesis import given, settings, strategies as st, HealthCheck
    R = ref.Removerter(base_params(scratch), write_files=False)

    def check(seed, n, alpha, mode, ties):
        rng = np.random.default_rng(seed)
        m = np.concatenate([rng.normal(0, 15, (n, 3)), rng.uniform(0, 1, (n, 1))], 1).astype(np.float32)
        if ties:
            m = np.concatenate([m, m[: n // 2]])
        K = 2
        scans = []
        for _ in range(K):
            ns = int(rng.integers(1, 300))
            scans.append(np.concatenate([rng.normal(0, 15, (ns, 3)), np.zeros((ns, 1))], 1).astype(np.float32))
        xyzi = np.concatenate(scans); off = np.concatenate([[0], np.cumsum([len(s) for s in scans])]).astype(np.int64)
        poses = np.stack([np.eye(4) for _ in range(K)])
        for k in range(K):
            a = rng.uniform(-np.pi, np.pi)
            poses[k][:3, :3] = [[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]]
            poses[k][:3, 3] = rng.normal(0, 5, 3)
        R.load_session_mem(0, xyzi, off, poses)
        R.load_session_mem(1, xyzi, off, poses)
        R.set_scans("keyframe_scans_static_projected_", xyzi, off, 1)
        inv = np.stack([ref.inverse4x4(p) for p in poses])
        rows, cols = oracle.reset_rimg_size(alpha)
        R.set_cloud(["map_global_curr_", "map_global_nd_", "map_global_pd_"][mode], m, 0)
        got = R.dynamic_idx(mode, 0, 1 if mode else 0, rows, cols, len(m))
        exp = oracle.remove_pass(m, xyzi, off, inv, [oracle.MODE_HD, oracle.MODE_ND, oracle.MODE_PD][mode], alpha, 0.1)
        assert values_equal(got, np.flatnonzero(exp))
    ref.rec.examples(check, lambda f: settings(max_examples=40, deadline=None, suppress_health_check=list(HealthCheck))(
        given(st.integers(0, 2**31 - 1), st.integers(3, 400), st.sampled_from([0.2, 0.5, 1.0, 2.5]), st.sampled_from([0, 1, 2]), st.booleans())(f)))
    R.close()


def test_property_knn_partition_matches_the_reference(scratch):
    """Property test: Session::extractLowDynPointsViaKnnDiff / extractHighDynPointsViaKnnDiff (Session.cpp:393-427, 487-504, 537-642) on random
    scans, targets, k, thresholds, poses and extrinsics: the coexist / diff partitions equal the oracle's knn_partition bit for bit (this covers
    the squared-distance mean, the double accumulate, the strict threshold and the base2lidar matrix the reference passes to local2global)."""
    from hypothesis import given, settings, strategies as st, HealthCheck

    def check(seed, k, thr, low, use_ext, order):
        rng = np.random.default_rng(seed)
        l2b = EXT if use_ext else np.eye(4)
        R = ref.Removerter(base_params(scratch, l2b), transform_order=order, write_files=False)
        K = 2
        scans = []
        for _ in range(K):
            ns = int(rng.integers(1, 400))
            scans.append(np.concatenate([rng.normal(0, 3, (ns, 3)), rng.uniform(0, 1, (ns, 1))], 1).astype(np.float32))
        xyzi = np.concatenate(scans); off = np.concatenate([[0], np.cumsum([len(s) for s in scans])]).astype(np.int64)
        poses = np.stack([np.eye(4) for _ in range(K)])
        for j in range(K):
            a = rng.uniform(-np.pi, np.pi)
            poses[j][:3, :3] = [[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]]
            poses[j][:3, 3] = rng.normal(0, 2, 3)
        nt = int(rng.integers(k, 600))
        target = np.concatenate([rng.normal(0, 3, (nt, 3)), np.zeros((nt, 1))], 1).astype(np.float32)
        # a few target points next to where the first scan lands in the map frame, so that both partitions are non-empty
        g = oracle.transform(oracle.transform(scans[0], oracle.inverse4x4(l2b), order), poses[0], order)
        m = min(nt, len(g), 50)
        target[:m, :3] = g[:m, :3] + rng.normal(0, 0.05, (m, 3)).astype(np.float32)
        R.load_session_mem(0, xyzi, off, poses)
        R.set_scans("keyframe_scans_static_projected_", xyzi, off, 0)
        R.extract_knn_diff(0, target, k, thr, low=low)
        if low:
            co, di = R.scans("scans_knn_coexist_", 0), R.scans("scans_knn_diff_", 0)
        else:
            co, di = None, R.scans("keyframe_scans_dynamic_", 0)
        for j in range(K):
            _, eco, edi = oracle.knn_partition(scans[j], poses[j], ref.inverse4x4(poses[j]), target, k, thr, lidar2base=l2b, order=order)
            assert bits_equal(di[j], edi), (j, "diff")
            if co is not None:
                assert bits_equal(co[j], eco), (j, "coexist")
        R.close()
    ref.rec.examples(check, lambda f: settings(max_examples=25, deadline=None, suppress_health_check=list(HealthCheck))(
        given(st.integers(0, 2**31 - 1), st.sampled_from([1, 2, 3]), st.sampled_from([0.01, 0.04, 0.5, 4.0]), st.booleans(), st.booleans(),
              st.sampled_from([0, 1]))(f)))


def test_property_keyframe_selection_and_pose_files_match_the_reference(tmp_path_factory, scratch):
    """Property test of the product's host logic (lt_mapper_b200/csrc/host/io.cpp) against the reference's Session::loadSessionInfo /
    parseKeyframes / parseKeyframesInROI (Session.cpp:80-118, 138-174, 230-263): random scan counts, index ranges (including empty and
    out-of-range ones), gaps, trajectories, and pose lines written in several number formats with 12 or 16 values."""
    from hypothesis import given, settings, strategies as st, HealthCheck
    counter = [0]

    def check(seed, nc, nq, start, end, gap):
        rng = np.random.default_rng(seed)
        counter[0] += 1
        root = str(tmp_path_factory.mktemp(f"kf{counter[0]}"))
        poses = {}
        for name, n in (("central", nc), ("query", nq)):
            os.makedirs(f"{root}/{name}/scans")
            P = np.stack([np.eye(4) for _ in range(n)])
            P[:, :3, 3] = np.cumsum(rng.normal(0, 3.0, (n, 3)), 0) + (rng.normal(0, 8, 3) if name == "query" else 0)
            poses[name] = P
            with open(f"{root}/{name}/poses.txt", "w") as f:
                for k in range(n):
                    open(f"{root}/{name}/scans/{k:06d}.pcd", "w").close()        # only the names matter before loadKeyframes
                    vals = P[k].ravel() if rng.random() < 0.3 else P[k][:3].ravel()   # 16 or 12 values per line (Session.cpp:106-108)
                    fmt = rng.integers(0, 3)
                    f.write(" ".join(repr(float(v)) if fmt == 0 else f"{v:.17e}" if fmt == 1 else f"{v:.17g}" for v in vals) + "\n")
        R = ref.Removerter(base_params(root, start_idx=start, end_idx=end, keyframe_gap=gap, save_pcd_directory=scratch + "/"), write_files=False)
        R.stage("loadSessionInfo"); R.stage("parseKeyframes")
        pc = removert.read_poses(f"{root}/central/poses.txt"); pq = removert.read_poses(f"{root}/query/poses.txt")
        assert bits_equal(pc, poses["central"]) and bits_equal(pq, poses["query"])
        exp_c = list(removert.parse_keyframes(nc, start, end, gap))
        assert R.keyframe_names(0) == [f"{k:06d}.pcd" for k in exp_c]
        kc = pc[exp_c].reshape(-1, 4, 4)
        assert bits_equal(R.keyframe_poses(0)[0], kc)
        exp_q = list(removert.parse_keyframes_in_roi(pq, kc, gap))
        assert R.keyframe_names(1) == [f"{k:06d}.pcd" for k in exp_q]
        R.close()
    ref.rec.examples(check, lambda f: settings(max_examples=40, deadline=None, suppress_health_check=list(HealthCheck))(
        given(st.integers(0, 2**31 - 1), st.integers(1, 40), st.integers(1, 40), st.integers(-3, 45), st.integers(-3, 45), st.integers(1, 7))(f)))


def test_points_on_pixel_boundaries_land_in_the_reference_pixel():
    """The most rounding-sensitive inputs: points whose azimuth / elevation sit on a pixel boundary (pre-round coordinate = n + 0.5) and their
    float neighbours a few ulps either side.  Each point is projected alone through the reference's map2RangeImg; the pixel it lands in (and
    the range stored there) must be the oracle's."""
    rng = np.random.default_rng(5)
    for (vfov, hfov, alpha), count in (((50.0, 360.0, 0.4), 1500), ((50.0, 360.0, 2.5), 400), ((33.2, 180.0, 1.0), 400)):
        rows, cols = oracle.reset_rimg_size(alpha, vfov, hfov)
        pts = []
        for _ in range(count):
            r = rng.uniform(0.5, 90.0)
            if rng.random() < 0.5:      # column boundary, arbitrary elevation inside the field of view
                az = np.deg2rad((rng.integers(0, cols) + 0.5) / cols * hfov - hfov / 2)
                el = np.deg2rad(rng.uniform(-vfov / 2, vfov / 2))
            else:                       # row boundary, arbitrary azimuth
                az = np.deg2rad(rng.uniform(-hfov / 2, hfov / 2))
                el = np.deg2rad(vfov / 2 - (rng.integers(0, rows) + 0.5) / rows * vfov)
            p = np.array([r * np.cos(el) * np.cos(az), r * np.cos(el) * np.sin(az), r * np.sin(el)], np.float32)
            for _ in range(int(rng.integers(0, 4))):   # walk a few ulps in a random coordinate
                j = int(rng.integers(0, 3))
                p[j] = np.nextafter(p[j], np.float32(np.inf if rng.random() < 0.5 else -np.inf))
            pts.append(p)
        pts = np.array(pts, np.float32)
        er, ec, erng = oracle.pixel_index(pts, rows, cols, vfov, hfov)
        first = np.array([[1.0, 0.0, 0.0, 0.0]], np.float32)     # index 0 is "no point" in the index image: keep a dummy there

        def landings():
            """Per point: (row, col, range bits) where the reference's map2RangeImg puts it."""
            out = []
            for p in pts:
                cloud = np.concatenate([first * 1e3, np.concatenate([p, [0.0]]).astype(np.float32)[None]])   # dummy far away at az = el = 0
                gr, gi = ref.compiled.map2rimg(cloud, rows, cols, vfov, hfov)
                rr, cc = np.argwhere(gi == 1)[0] if (gi == 1).any() else (-1, -1)
                out.append((rr, cc, gr[rr, cc].view(np.uint32)))
            return np.array(out, np.int64)
        got = ref.capture("map2rimg landings", (pts, rows, cols, vfov, hfov), landings)
        assert len(got) == count
        assert values_equal(got, np.stack([er, ec, erng.view(np.uint32)], 1).astype(np.int64))


def test_full_size_scans_match_the_reference(scratch):
    """BASELINE-sized scans (64 x 1800 rays, ~103 k returns each), 3 keyframes per session, the bench's schedule and kNN setting: every
    cloud the compiled reference holds after Steps 0-2 equals the oracle's (the dense, full-resolution counterpart of the small-scene tests)."""
    import synth
    sched = [(0, 2.5), (0, 2.0), (0, 1.5), (1, 1.0)]
    pair = synth.make_pair(3)
    R = ref.Removerter(base_params(scratch, num_nn_points_within=1, dist_nn_points_within=0.04), write_files=False)
    O = oracle.Removerter(schedule=sched, num_knn=1, knn_thr=0.04, threads=8)
    for s, d in enumerate(pair):
        R.load_session_mem(s, d.xyzi, d.offsets, d.poses)
        O.load_session(s, d.xyzi, d.offsets, d.poses, np.stack([ref.inverse4x4(p) for p in d.poses]))
    for st in ("precleaningKeyframes", "makeGlobalMap"):
        R.stage(st); O.stage(st)
    R.high_dyn_with_schedule(sched)
    O.stage("removeHighDynamicPoints")
    for st in ("parseStaticScansViaProjection", "detectLowDynamicPoints"):
        R.stage(st); O.stage(st)
    for s in (0, 1):
        for name in ("map_global_orig_", "map_global_curr_", "map_global_curr_static_", "map_global_curr_dynamic_", "map_global_nd_", "map_global_nd_strong_",
                     "map_global_nd_weak_", "map_global_pd_", "map_global_pd_strong_", "map_global_pd_weak_"):
            assert bits_equal(R.cloud(name, s), O.cloud(name, s)), (name, s)
        for name in ("keyframe_scans_", "keyframe_scans_dynamic_", "keyframe_scans_static_projected_", "scans_knn_coexist_", "scans_knn_diff_"):
            got, exp = R.scans(name, s), O.clouds(name, s)
            assert len(got) == len(exp) == 3 and all(bits_equal(a, b) for a, b in zip(got, exp)), (name, s)
    assert len(R.cloud("map_global_orig_", 0)) > 250000 and len(R.cloud("map_global_curr_dynamic_", 0)) > 0
    R.close()
