"""File-level surface (yaml, poses, PCD, keyframe selection, pcl::VoxelGrid) -- host logic, CPU only."""
import os

import numpy as np
import pytest

from lt_mapper_b200 import removert

REF_YAML = os.path.join(os.path.dirname(__file__), "golden", "params_ltmapper.yaml")      # the reference's shipped ltremovert/config/params_ltmapper.yaml


def test_pcd_roundtrip_and_layout(tmp_path):
    rng = np.random.default_rng(0)
    pts = rng.normal(size=(1000, 4)).astype(np.float32)
    for octree in (False, True):
        p = str(tmp_path / f"a{int(octree)}.pcd")
        removert.write_pcd(p, pts, octree_layout=octree)
        assert np.array_equal(removert.read_pcd(p), pts)
        hdr = open(p, "rb").read(400).decode("latin1")
        assert "FIELDS x y z intensity" in hdr and "SIZE 4 4 4 4" in hdr and "TYPE F F F F" in hdr and "DATA binary" in hdr
        assert ("WIDTH 1\nHEIGHT 1000" in hdr) == octree and ("WIDTH 1000\nHEIGHT 1" in hdr) == (not octree)   # utility.cpp:217-218
    # ascii PCD with extra fields in a different order (what other savers write)
    p = str(tmp_path / "b.pcd")
    with open(p, "w") as f:
        f.write("# .PCD v0.7\nVERSION 0.7\nFIELDS intensity x y z ring\nSIZE 4 4 4 4 2\nTYPE F F F F U\nCOUNT 1 1 1 1 1\nWIDTH 2\nHEIGHT 1\nPOINTS 2\nDATA ascii\n")
        f.write("7 1.5 2.5 3.5 4\n8 -1 -2 -3 5\n")
    assert np.array_equal(removert.read_pcd(p), np.array([[1.5, 2.5, 3.5, 7], [-1, -2, -3, 8]], np.float32))
    with pytest.raises(IOError):
        removert.read_pcd(str(tmp_path / "missing.pcd"))


def test_pose_file(tmp_path):
    p = str(tmp_path / "poses.txt")
    T = np.arange(12, dtype=np.float64).reshape(3, 4) * 0.5
    with open(p, "w") as f:
        f.write(" ".join(repr(float(v)) for v in T.ravel()) + "\n")
        f.write(" ".join(repr(float(v)) for v in np.eye(4).ravel()) + "\n")
    P = removert.read_poses(p)
    assert P.shape == (2, 4, 4)
    assert np.array_equal(P[0][:3], T) and np.array_equal(P[0][3], [0, 0, 0, 1])   # Session.cpp:106-108
    assert np.array_equal(P[1], np.eye(4))


def test_parse_keyframes_quirk():
    # Session.cpp:138-174: an out-of-range index also skips its successor, so from 0 the loop visits 0, 2, 4, ... until inside
    # the range; inside, every `gap`-th VALID index is taken.
    assert list(removert.parse_keyframes(20, 5, 12, 1)) == [6, 7, 8, 9, 10, 11, 12]      # 0,2,4 skipped in pairs -> enters at 6, not 5
    assert list(removert.parse_keyframes(20, 4, 12, 1)) == [4, 5, 6, 7, 8, 9, 10, 11, 12]
    assert list(removert.parse_keyframes(20, 4, 12, 3)) == [4, 7, 10]
    assert list(removert.parse_keyframes(10, 0, 100, 2)) == [0, 2, 4, 6, 8]
    # after the range: 13 is out -> skip 14 too, 15 out -> skip 16 ...
    assert list(removert.parse_keyframes(6, 1, 2, 1)) == [2]                            # idx 0 out (skips 1), 2 in, 3 out (skips 4), 5 out


def test_parse_keyframes_in_roi():
    def pose(x, y):
        T = np.eye(4); T[0, 3] = x; T[1, 3] = y
        return T
    scans = [pose(x, 0) for x in range(0, 40, 2)]
    roi = [pose(10, 0), pose(12, 3)]
    got = removert.parse_keyframes_in_roi(scans, roi, 1)
    exp = [i for i, s in enumerate(scans) if min(np.linalg.norm(s[:3, 3] - r[:3, 3]) for r in roi) <= 10.0]
    assert list(got) == exp
    assert list(removert.parse_keyframes_in_roi(scans, roi, 2)) == exp[::2]


def test_voxel_grid_overflow_and_centroids():
    rng = np.random.default_rng(1)
    # outdoor-sized scan at 0.05 m: (dx*dy*dz) overflows int32 -> PCL returns the input unchanged (Session.cpp:284-289 + PCL warning)
    big = rng.uniform(-90, 90, (5000, 4)).astype(np.float32)
    out, ov = removert.voxel_grid(big, 0.05)
    assert ov and np.array_equal(out, big)
    # small extent: real voxelisation; compare with an independent numpy restatement
    pts = rng.uniform(-2, 2, (20000, 4)).astype(np.float32)
    leaf = np.float32(0.25)
    out, ov = removert.voxel_grid(pts, float(leaf))
    assert not ov
    inv = np.float32(1.0) / leaf
    mn = np.floor(pts[:, :3].min(0) * inv).astype(np.int64)
    mx = np.floor(pts[:, :3].max(0) * inv).astype(np.int64)
    div = mx - mn + 1
    ijk = (np.floor(pts[:, :3] * inv) - mn.astype(np.float32)).astype(np.int64)
    idx = ijk[:, 0] + ijk[:, 1] * div[0] + ijk[:, 2] * div[0] * div[1]
    assert len(out) == len(np.unique(idx))
    order = np.argsort(idx, kind="stable")
    first = np.flatnonzero(np.diff(idx[order], prepend=-1))
    # voxel order is ascending idx; centroids agree with the per-voxel mean to f32 summation-order error
    mean = np.add.reduceat(pts[order].astype(np.float64), first, axis=0) / np.diff(np.append(first, len(pts)))[:, None]
    assert np.allclose(out, mean, atol=2e-5)


def test_voxel_grid_scans_equals_scan_by_scan():
    """The batched load-time filter (cascade promotion) == the per-scan filter, bit for bit: pass-through scans (PCL's overflow exit),
    really voxelised scans, an empty scan and a one-point scan, in one session."""
    rng = np.random.default_rng(7)
    scans = [rng.uniform(-90, 90, (4000, 4)).astype(np.float32),            # overflow exit
             rng.uniform(-3, 3, (30000, 4)).astype(np.float32),             # voxelised (many points per voxel: summation order matters)
             np.zeros((0, 4), np.float32),
             rng.uniform(-1, 1, (1, 4)).astype(np.float32),
             rng.normal(0, 0.4, (15000, 4)).astype(np.float32),             # dense cluster
             rng.uniform(-80, 80, (2500, 4)).astype(np.float32)]            # overflow exit again (last scan)
    off = np.concatenate([[0], np.cumsum([len(s) for s in scans])]).astype(np.int64)
    allp = np.concatenate(scans)
    for leaf in (0.05, 0.3):
        got, got_off = removert.voxel_grid_scans(allp, off, leaf)
        exp = [removert.voxel_grid(s, leaf) for s in scans]
        assert [int(x) for x in np.diff(got_off)] == [len(e[0]) for e in exp]
        assert [bool(e[1]) for e in exp] == ([True, False, False, False, False, True] if leaf == 0.05 else [False] * 6)   # mix of both exits
        for k, (e, _) in enumerate(exp):
            assert np.array_equal(got[got_off[k]:got_off[k + 1]].view(np.uint32), e.view(np.uint32)), (leaf, k)
    # all scans pass through: output == input
    got, got_off = removert.voxel_grid_scans(np.concatenate([scans[0], scans[5]]), np.array([0, 4000, 6500]), 0.05)
    assert np.array_equal(got_off, [0, 4000, 6500]) and np.array_equal(got, np.concatenate([scans[0], scans[5]]))
    # no scans at all
    got, got_off = removert.voxel_grid_scans(np.zeros((0, 4), np.float32), np.array([0]), 0.05)
    assert len(got) == 0 and list(got_off) == [0]


def test_yaml_reader(tmp_path):
    p = str(tmp_path / "params.yaml")
    with open(p, "w") as f:
        f.write('removert:\n\n  # comment\n  saveMapPCD: true \n  save_pcd_directory: "/tmp/out dir/" # trailing\n  sequence_vfov: 50 # deg\n'
                '  ExtrinsicLiDARtoPoseBase: [1.0, 0.0, 0.0, 0.0, \n                             0.0, 1.0, 0.0, 0.0, \n'
                '                             0.0, 0.0, 1.0, 0.0, \n                             0.0, 0.0, 0.0, 1.0]\n'
                '  remove_resolution_list: [2.5, 2.0, 1.5] # list\n  num_nn_points_within: 2\n  dist_nn_points_within: 0.01\n')
    assert removert.yaml_get(p, "removert/saveMapPCD")[0] == "true"
    assert removert.yaml_get(p, "removert/save_pcd_directory")[0] == "/tmp/out dir/"
    assert removert.yaml_get(p, "removert/sequence_vfov")[0] == "50"
    assert list(removert.yaml_get(p, "removert/ExtrinsicLiDARtoPoseBase")[1]) == list(np.eye(4).ravel())
    assert list(removert.yaml_get(p, "removert/remove_resolution_list")[1]) == [2.5, 2.0, 1.5]
    assert removert.yaml_get(p, "removert/dist_nn_points_within")[0] == "0.01"


def test_yaml_reader_on_the_reference_config():
    assert removert.yaml_get(REF_YAML, "removert/start_idx")[0] == "1100"
    assert removert.yaml_get(REF_YAML, "removert/keyframe_gap")[0] == "1"
    assert removert.yaml_get(REF_YAML, "removert/num_nn_points_within")[0] == "2"
    assert list(removert.yaml_get(REF_YAML, "removert/remove_resolution_list")[1]) == [2.5]
    assert list(removert.yaml_get(REF_YAML, "removert/ExtrinsicLiDARtoPoseBase")[1]) == list(np.eye(4).ravel())
    assert removert.yaml_get(REF_YAML, "removert/saveMapPCD")[0] == "true"


def _lzf_compress(data: bytes) -> bytes:
    """A valid (not optimal) liblzf stream: greedy back references to the previous occurrence of a 3-byte prefix, literals otherwise."""
    out = bytearray(); lit = bytearray(); last = {}
    i, n = 0, len(data)

    def flush():
        nonlocal lit
        for s in range(0, len(lit), 32):
            chunk = lit[s:s + 32]
            out.append(len(chunk) - 1); out.extend(chunk)
        lit = bytearray()
    while i < n:
        key = data[i:i + 3]
        ref = last.get(key) if len(key) == 3 else None
        if ref is not None and 0 < i - ref <= 8192:
            ln = 3
            while i + ln < n and ln < 264 and data[ref + ln] == data[i + ln]:
                ln += 1
            flush()
            dist = i - ref - 1
            l2 = ln - 2
            if l2 < 7:
                out.append((l2 << 5) | (dist >> 8))
            else:
                out.append((7 << 5) | (dist >> 8)); out.append(l2 - 7)
            out.append(dist & 0xff)
            for j in range(i, i + ln):
                last[data[j:j + 3]] = j
            i += ln
        else:
            last[key] = i
            lit.append(data[i]); i += 1
    flush()
    return bytes(out)


def test_pcd_binary_compressed(tmp_path):
    """pcl::io::loadPCDFile (Session.cpp:275) also accepts DATA binary_compressed: LZF stream of a FIELD-MAJOR payload."""
    import struct
    rng = np.random.default_rng(3)
    n = 5000
    pts = rng.normal(size=(n, 4)).astype(np.float32)
    pts[:, 3] = np.repeat(np.arange(n // 50, dtype=np.float32), 50)          # long runs -> back references incl. overlapping ones
    extra = rng.normal(size=n).astype(np.float32)                            # an extra field between z and intensity is skipped
    payload = pts[:, 0].tobytes() + pts[:, 1].tobytes() + pts[:, 2].tobytes() + extra.tobytes() + pts[:, 3].tobytes()
    comp = _lzf_compress(payload)
    assert len(comp) < len(payload)
    hdr = (f"# .PCD v0.7 - Point Cloud Data file format\nVERSION 0.7\nFIELDS x y z ring intensity\nSIZE 4 4 4 4 4\nTYPE F F F F F\nCOUNT 1 1 1 1 1\n"
           f"WIDTH {n}\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS {n}\nDATA binary_compressed\n").encode()
    p = tmp_path / "c.pcd"
    p.write_bytes(hdr + struct.pack("<II", len(comp), len(payload)) + comp)
    got = removert.read_pcd(str(p))
    assert np.array_equal(got.view(np.uint32), pts.view(np.uint32))
    # truncated stream -> error, not garbage
    p.write_bytes(hdr + struct.pack("<II", len(comp), len(payload)) + comp[:-7])
    with pytest.raises(IOError):
        removert.read_pcd(str(p))


def test_inverse_poses_is_the_cofactor_inverse_of_the_oracle():
    """ltrh_invert_poses == the oracle's / reference shim's Eigen::Matrix4d::inverse() stand-in, bit for bit (an LU inverse is not)."""
    import oracle
    import synth
    d = synth.make_session(1, 64, beams=4, az_steps=8)
    assert np.array_equal(removert.inverse_poses(d.poses), oracle.inverse_poses(d.poses))
