"""File-in/file-out drop-in: apps/ltremovert_b200 on a synthetic dataset on disk == the oracle pipeline on the same keyframes."""
import os
import subprocess

import numpy as np
import pytest

import oracle
from lt_mapper_b200 import removert
from oracle import ref as ref_lib
from oracle.ref_golden import RecordedRef, bits_equal

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "lt_mapper_b200", "ltremovert_b200")
# the reference runs' output trees, replayed from tests/golden/ref_driver.json.gz (oracle/ref_golden.py); to record them where oracle/_ref is
# built:  LTR_RECORD_REFERENCE=1 python -m pytest -p no:xdist tests/test_gpu_driver.py
REF = RecordedRef(os.path.join(os.path.dirname(__file__), "golden", "ref_driver.json.gz"))


@pytest.fixture(scope="module")
def _ref_recording(request):
    yield
    REF.rec.save(request.session.testsfailed == 0)


@pytest.fixture
def reference(request, _ref_recording):
    with REF.rec.test(request.node.name):
        yield REF


def _tree(d):
    return sorted(os.path.relpath(os.path.join(p, f), d) for p, _, fs in os.walk(d) for f in fs)


def _read_tree(d):
    return {f: removert.read_pcd(str(d / f)) for f in _tree(d)}


def _write_session(d, sess):
    os.makedirs(d / "Scans", exist_ok=True)
    with open(d / "poses.txt", "w") as f:
        for k in range(sess.K):
            removert.write_pcd(str(d / "Scans" / f"{k:06d}.pcd"), sess.scan(k))
            f.write(" ".join(repr(float(v)) for v in sess.poses[k][:3].ravel()) + "\n")


def test_driver_matches_oracle(tmp_path, small_pair):
    c, q = small_pair
    _write_session(tmp_path / "central", c)
    _write_session(tmp_path / "query", q)
    out = tmp_path / "out"
    cfg = tmp_path / "params.yaml"
    cfg.write_text(f"""removert:
  saveMapPCD: true
  save_pcd_directory: "{out}"
  central_sess_scan_dir: "{tmp_path}/central/Scans/"
  central_sess_pose_path: "{tmp_path}/central/poses.txt"
  query_sess_scan_dir: "{tmp_path}/query/Scans/"
  query_sess_pose_path: "{tmp_path}/query/poses.txt"
  sequence_vfov: 50
  sequence_hfov: 360
  ExtrinsicLiDARtoPoseBase: [1.0, 0.0, 0.0, 0.0,
                             0.0, 1.0, 0.0, 0.0,
                             0.0, 0.0, 1.0, 0.0,
                             0.0, 0.0, 0.0, 1.0]
  keyframe_gap: 1
  start_idx: 2
  end_idx: 5
  remove_resolution_list: [2.5]
  downsample_voxel_size: 0.05
  num_nn_points_within: 2
  dist_nn_points_within: 0.01
""")
    r = subprocess.run([BIN, "--config", str(cfg)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    # the same keyframe selection through the host helpers, then the oracle pipeline
    kc = removert.parse_keyframes(c.K, 2, 5, 1)
    assert list(kc) == [2, 3, 4, 5]
    kq = removert.parse_keyframes_in_roi(q.poses, c.poses[kc], 1)
    O = oracle.Removerter(num_knn=2, knn_thr=0.01)
    for s, d, ks in ((0, c, kc), (1, q, kq)):
        xyzi = np.concatenate([d.scan(k) for k in ks]); off = np.concatenate([[0], np.cumsum([len(d.scan(k)) for k in ks])])
        poses = removert.read_poses(str(tmp_path / ("central" if s == 0 else "query") / "poses.txt"))[ks]
        O.load_session(s, xyzi, off, poses, oracle.inverse_poses(poses))
    O.run(step3=True)
    for name in ["OriginalNoisyCentralMapGlobal", "central_sess_high_dyn", "query_sess_high_dyn", "union_map_queryside", "union_map_centralside",
                 "pd_map", "nd_map", "strong_nd_map", "weak_nd_map", "strong_pd_map", "weak_pd_map", "updated_map", "updated_map_strong"]:
        got = removert.read_pcd(str(out / (name + ".pcd")))
        exp = O.cloud("saved:" + name)
        assert got.shape == exp.shape and np.array_equal(got.view(np.uint32), exp.view(np.uint32)), name
    for d, member in (("scans_updated", "keyframe_scans_updated_"), ("scans_updated_strong", "keyframe_scans_updated_strong_"), ("scans_pd", "keyframe_scans_pd_"),
                      ("scans_pd_strong", "keyframe_scans_strong_pd_"), ("scans_nd_strong", "keyframe_scans_strong_nd_")):
        files = sorted(os.listdir(out / d))
        assert files == [f"{k:06d}.pcd" for k in kc]          # per-keyframe files keep the input scan's name (Removerter.cpp:1642-1645)
        for i, fn in enumerate(files):
            got = removert.read_pcd(str(out / d / fn))
            exp = O.cloud(member, 0, i)
            assert got.shape == exp.shape and np.array_equal(got.view(np.uint32), exp.view(np.uint32)), (d, fn)
    assert os.path.isdir(out / "map_static") and os.path.isdir(out / "map_dynamic")


def test_driver_matches_compiled_reference(tmp_path, small_pair, reference):
    """The same dataset and parameters through (a) the reference's own Removerter::run(), compiled behind the third-party stand-ins
    (oracle/_ref, see oracle/ref_shim; its output tree is replayed), and (b) the drop-in binary: identical output trees."""
    c, q = small_pair
    _write_session(tmp_path / "central", c)
    _write_session(tmp_path / "query", q)
    ext = [0.955336489125606, -0.29552020666133955, 0.0, 0.5, 0.29552020666133955, 0.955336489125606, 0.0, -0.2, 0.0, 0.0, 1.0, 1.1, 0.0, 0.0, 0.0, 1.0]
    common = dict(sequence_vfov=50.0, sequence_hfov=360.0, keyframe_gap=2, start_idx=0, end_idx=5, downsample_voxel_size=0.05,
                  num_nn_points_within=1, dist_nn_points_within=0.04)
    out_ref, out_gpu = tmp_path / "out_ref", tmp_path / "out_gpu"

    def run_ref():
        R = reference.compiled.Removerter(dict(common, saveMapPCD=True, save_pcd_directory=str(out_ref), ExtrinsicLiDARtoPoseBase=ext,
                                               central_sess_scan_dir=f"{tmp_path}/central/Scans/", central_sess_pose_path=f"{tmp_path}/central/poses.txt",
                                               query_sess_scan_dir=f"{tmp_path}/query/Scans/", query_sess_pose_path=f"{tmp_path}/query/poses.txt"))
        R.run()
        R.close()
        return _read_tree(out_ref)
    ref_out = reference.capture("reference run", ([(d.xyzi, d.offsets, d.poses) for d in small_pair], ext, common), run_ref)
    cfg = tmp_path / "params.yaml"
    cfg.write_text("removert:\n  saveMapPCD: true\n" + f'  save_pcd_directory: "{out_gpu}"\n'
                   + f'  central_sess_scan_dir: "{tmp_path}/central/Scans/"\n  central_sess_pose_path: "{tmp_path}/central/poses.txt"\n'
                   + f'  query_sess_scan_dir: "{tmp_path}/query/Scans/"\n  query_sess_pose_path: "{tmp_path}/query/poses.txt"\n'
                   + "  ExtrinsicLiDARtoPoseBase: [" + ", ".join(repr(v) for v in ext) + "]\n"
                   + "".join(f"  {k}: {v}\n" for k, v in common.items()))
    r = subprocess.run([BIN, "--config", str(cfg)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr

    files = sorted(ref_out)
    assert files == _tree(out_gpu) and len(files) >= 14 + 5 * 3
    for f in files:
        assert bits_equal(ref_out[f], removert.read_pcd(str(out_gpu / f))), f


def test_cascade_through_files_matches_compiled_reference(tmp_path, reference):
    """Multi-session cascade the way the reference does it (SURVEY §8f): a run's scans_updated/ + the central poses become the next
    run's central session, diffed against a third session.  Both implementations consume their OWN first-run outputs; the second-run
    output trees must still be identical (LT-map composition error would compound here)."""
    import shutil
    import synth
    K = 4
    sessions = [synth.make_session(s, K, beams=32, az_steps=900) for s in (0, 1, 2)]
    for name, s in zip("abc", sessions):
        _write_session(tmp_path / name, s)
    common = dict(sequence_vfov=50.0, sequence_hfov=360.0, keyframe_gap=1, start_idx=0, end_idx=100, downsample_voxel_size=0.05,
                  num_nn_points_within=2, dist_nn_points_within=0.01)
    ident = [1.0, 0.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 0.0, 1.0]

    def run_ref(central_scans, query, out):
        R = reference.compiled.Removerter(dict(common, saveMapPCD=True, save_pcd_directory=str(out), ExtrinsicLiDARtoPoseBase=ident,
                                central_sess_scan_dir=str(central_scans), central_sess_pose_path=f"{tmp_path}/a/poses.txt",
                                query_sess_scan_dir=f"{tmp_path}/{query}/Scans/", query_sess_pose_path=f"{tmp_path}/{query}/poses.txt"))
        R.run()
        R.close()

    def run_gpu(central_scans, query, out):
        cfg = tmp_path / f"params_{query}.yaml"
        cfg.write_text("removert:\n  saveMapPCD: true\n" + f'  save_pcd_directory: "{out}"\n'
                       + f'  central_sess_scan_dir: "{central_scans}"\n  central_sess_pose_path: "{tmp_path}/a/poses.txt"\n'
                       + f'  query_sess_scan_dir: "{tmp_path}/{query}/Scans/"\n  query_sess_pose_path: "{tmp_path}/{query}/poses.txt"\n'
                       + "  ExtrinsicLiDARtoPoseBase: [" + ", ".join(repr(v) for v in ident) + "]\n"
                       + "".join(f"  {k}: {v}\n" for k, v in common.items()))
        r = subprocess.run([BIN, "--config", str(cfg)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr

    def cascade(tag, run):
        run(tmp_path / "a" / "Scans", "b", tmp_path / f"{tag}1")
        nxt = tmp_path / f"{tag}_central2"
        shutil.copytree(tmp_path / f"{tag}1" / "scans_updated", nxt)
        run(nxt, "c", tmp_path / f"{tag}2")
        return {stage: _read_tree(tmp_path / f"{tag}{stage}") for stage in ("1", "2")}
    ref_out = reference.capture("reference cascade", ([(s.xyzi, s.offsets, s.poses) for s in sessions], common), lambda: cascade("ref", run_ref))
    cascade("gpu", run_gpu)
    for stage in ("1", "2"):
        b = tmp_path / ("gpu" + stage)
        files = sorted(ref_out[stage])
        assert files == _tree(b) and len(files) >= 14 + 5 * K
        for f in files:
            assert bits_equal(ref_out[stage][f], removert.read_pcd(str(b / f))), (stage, f)
    assert len(removert.read_pcd(str(tmp_path / "gpu2" / "nd_map.pcd"))) > 0 and len(removert.read_pcd(str(tmp_path / "gpu2" / "pd_map.pcd"))) > 0


@pytest.mark.skipif(not ref_lib.available("dropin"), reason="oracle/_ref/libltremovert_dropin.so not built (needs the reference's sources)")
def test_reference_node_with_b200_core(tmp_path, small_pair, reference):
    """INTEGRATION.md "B" executed: the reference's own Removerter object keeps its loaders (loadSessionInfo, parseKeyframes, loadKeyframes)
    and writers (saveAllTypeOfScans, savePCDFileBinary); Steps 0-3 run on libltr_removert.so / libltr_b200.so through
    include/ltr_pcl_adapter.hpp (oracle/ref_shim/dropin_capi.cpp).  The files it writes equal the files of the unmodified reference run
    (replayed).  The drop-in library holds the reference's own sources, so it exists only where they were available to build it."""
    c, q = small_pair
    _write_session(tmp_path / "central", c)
    _write_session(tmp_path / "query", q)
    ext = [0.955336489125606, -0.29552020666133955, 0.0, 0.5, 0.29552020666133955, 0.955336489125606, 0.0, -0.2, 0.0, 0.0, 1.0, 1.1, 0.0, 0.0, 0.0, 1.0]

    def params(out):
        return dict(sequence_vfov=50.0, sequence_hfov=360.0, keyframe_gap=1, start_idx=1, end_idx=4, downsample_voxel_size=0.05,
                    num_nn_points_within=2, dist_nn_points_within=0.01, saveMapPCD=True, save_pcd_directory=str(out), ExtrinsicLiDARtoPoseBase=ext,
                    central_sess_scan_dir=f"{tmp_path}/central/Scans/", central_sess_pose_path=f"{tmp_path}/central/poses.txt",
                    query_sess_scan_dir=f"{tmp_path}/query/Scans/", query_sess_pose_path=f"{tmp_path}/query/poses.txt")
    out_ref, out_b200 = tmp_path / "out_ref", tmp_path / "out_b200"

    def run_ref():
        R = reference.compiled.Removerter(params(out_ref), transform_order=1)
        R.run()
        R.close()
        return _read_tree(out_ref)
    ref_out = reference.capture("reference run", ([(d.xyzi, d.offsets, d.poses) for d in small_pair], ext), run_ref)
    D = ref_lib.Removerter(params(out_b200), transform_order=1, omp="dropin")
    D.dropin_run(transform_order=1)
    D.close()

    files = sorted(ref_out)
    assert files == _tree(out_b200) and len(files) >= 14 + 5 * 3
    for f in files:
        assert bits_equal(ref_out[f], removert.read_pcd(str(out_b200 / f))), f
