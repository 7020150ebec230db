"""Key-frame files (SURVEY.md section 8f row N3, the on-disk format): lsd_keyframe_save / lsd_keyframe_load and the pybind
`dump_keyframe` against the reference's own KeyFrame::save / loadOdom / loadPcd compiled unmodified (oracle/ref_keyframe.cpp
-> oracle/_ref/libref_keyframe.so) and against the PCD reader the reference vendors (third_party/pypcd.py), through what
those wrote and read on the same seeded inputs (tests/golden/keyframe_ref.npz, tests/golden/make_golden_keyframe.py).
Host-only code: runs without a GPU."""
import hashlib
import os
import sys

import numpy as np
import pytest

import lsdreg

_HERE = os.path.dirname(os.path.abspath(__file__))
_GOLD = os.path.join(_HERE, "golden", "keyframe_ref.npz")


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(_GOLD))


def _sha(b) -> str:
    return hashlib.sha256(b if isinstance(b, bytes) else np.ascontiguousarray(b).tobytes()).hexdigest()


def _poses(rng):
    from lsdreg import synth
    out = [np.eye(4)]
    for k in range(6):
        T = np.eye(4)
        T[:3, :3] = synth.rot_from_rpy(*rng.uniform(-3, 3, 3))
        T[:3, 3] = rng.uniform(-1, 1, 3) * 10.0 ** rng.integers(-7, 6)      # 1e-7 .. 1e5: fixed and scientific notation, all widths
        out.append(T)
    out.append(np.array([[1, 0, 0, -123456.789], [0, 1, 0, 1e-9], [0, 0, 1, 3.0], [0, 0, 0, 1.0]]))
    return out


def _cloud(rng, n):
    p = np.zeros((n, 4), np.float32)
    p[:, :3] = rng.uniform(-80, 80, (n, 3)); p[:, 3] = rng.uniform(0, 1, n)
    return p


def test_files_equal_the_reference_writers_byte_for_byte(tmp_path, gold):
    rng = np.random.default_rng(4)
    for k, T in enumerate(_poses(rng)):
        pts = _cloud(rng, 1000 + 37 * k)
        stamp, kid = 1_695_000_000_000_000 + 123_456 * k + 7, 40 + k
        a = tmp_path / f"ours{k}"
        a.mkdir()
        lsdreg.keyframe_save(str(a), stamp, kid, pts, T)
        ref_data = gold[f"save{k}_data"].tobytes()
        assert (a / "data").read_bytes() == ref_data, ref_data.decode()
        assert _sha((a / "cloud.pcd").read_bytes()) == gold["save_pcd_sha256"][k]
        assert sorted(os.listdir(a)) == ["cloud.pcd", "data"]


def test_each_side_loads_what_the_other_wrote(tmp_path, gold):
    rng = np.random.default_rng(5)
    for k, T in enumerate(_poses(rng)[:4]):
        pts = _cloud(rng, 500 + k)
        stamp, kid = 1_700_000_000_000_000 + 999_999 - k, 7 + k
        a, b = tmp_path / f"ours{k}", tmp_path / f"ref{k}"
        a.mkdir(); b.mkdir()
        lsdreg.keyframe_save(str(a), stamp, kid, pts, T)
        (b / "data").write_bytes(gold[f"load{k}_data"].tobytes())
        (b / "cloud.pcd").write_bytes(gold[f"load{k}_pcd"].tobytes())
        # ours <- reference's files
        s1, i1, T1, p1 = lsdreg.keyframe_load(str(b))
        # reference <- our files: the reference read its own files, and ours are the same bytes
        assert (a / "data").read_bytes() == (b / "data").read_bytes() and (a / "cloud.pcd").read_bytes() == (b / "cloud.pcd").read_bytes()
        s2, i2, T2, n2 = int(gold["load_stamp"][k]), int(gold["load_id"][k]), gold["load_T"][k], int(gold["load_n"][k])
        assert n2 == pts.shape[0] == p1.shape[0]
        assert s1 == s2 == stamp and i1 == i2 == kid
        np.testing.assert_array_equal(T1, T2)
        np.testing.assert_allclose(T1, T, rtol=1e-5, atol=1e-12)          # six significant digits survive the text file
        assert _sha(np.ascontiguousarray(p1, np.float32)) == gold["load_pts_sha256"][k]      # p1 == what the reference loaded
        np.testing.assert_array_equal(p1[:, :3], pts[:, :3])
        np.testing.assert_allclose(p1[:, 3], pts[:, 3], rtol=3e-7)        # x 255 then / 255 in fp32


def test_round_trip_empty_cloud_and_errors(tmp_path):
    rng = np.random.default_rng(6)
    d = tmp_path / "kf"; d.mkdir()
    T = np.eye(4); T[:3, 3] = [1.5, -2.25, 0.125]
    pts = _cloud(rng, 321)
    lsdreg.keyframe_save(str(d), 12_345_678, 3, pts, T)
    assert (d / "data").read_text() == "stamp 12 345678000\nestimate\n    1     0     0   1.5\n    0     1     0 -2.25\n    0     0     1 0.125\n    0     0     0     1\n" \
                                       "odom \n    1     0     0   1.5\n    0     1     0 -2.25\n    0     0     1 0.125\n    0     0     0     1\nid 3\n"
    head = (d / "cloud.pcd").read_bytes()[:200].decode("ascii", "replace")
    assert head.startswith("# .PCD v0.7 - Point Cloud Data file format\nVERSION 0.7\nFIELDS x y z intensity\nSIZE 4 4 4 4\nTYPE F F F F\nCOUNT 1 1 1 1\nWIDTH 321\nHEIGHT 1\n"
                           "VIEWPOINT 0 0 0 1 0 0 0\nPOINTS 321\nDATA binary\n")
    assert os.path.getsize(d / "cloud.pcd") == len(head.split("DATA binary\n")[0]) + len("DATA binary\n") + 321 * 16
    s, i, T1, p = lsdreg.keyframe_load(str(d))
    assert (s, i) == (12_345_678, 3)
    np.testing.assert_array_equal(T1, T)
    np.testing.assert_array_equal(p[:, :3], pts[:, :3])
    # an empty key frame gets the reference's ASCII stub (slam/common/pcd_writer.cpp) and loads as zero points
    e = tmp_path / "empty"; e.mkdir()
    lsdreg.keyframe_save(str(e), 1, 0, np.zeros((0, 4), np.float32), T)
    assert (e / "cloud.pcd").read_text().endswith("WIDTH 0\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS 0\nDATA ascii\n")
    assert lsdreg.keyframe_load(str(e))[3].shape == (0, 4)
    with pytest.raises(lsdreg.LsdError):
        lsdreg.keyframe_save(str(tmp_path / "does_not_exist"), 1, 0, pts, T)
    with pytest.raises(lsdreg.LsdError):
        lsdreg.keyframe_load(str(tmp_path / "does_not_exist"))
    (e / "cloud.pcd").write_text("# .PCD v0.7\nFIELDS x y z\nSIZE 4 4 4\nTYPE F F F\nPOINTS 1\nDATA ascii\n0 0 0\n")
    with pytest.raises(lsdreg.LsdError):
        lsdreg.keyframe_load(str(e))


def test_pybind_dump_keyframe_writes_the_same_files(tmp_path):
    sys.path.insert(0, os.path.join(os.path.dirname(_HERE), "lidar-slam-detection_b200"))
    import slam_wrapper
    rng = np.random.default_rng(7)
    pts = _cloud(rng, 200)
    T = _poses(rng)[2].astype(np.float32)                    # the reference binding takes float32 arrays (py_utils.cpp:82-90)
    a, b = tmp_path / "a", tmp_path / "b"
    a.mkdir(); b.mkdir()
    slam_wrapper.dump_keyframe(str(a), 1_700_000_000_123_456, 12, pts, T)
    lsdreg.keyframe_save(str(b), 1_700_000_000_123_456, 12, pts, T.astype(np.float64))
    for f in ("data", "cloud.pcd"):
        assert (a / f).read_bytes() == (b / f).read_bytes()


def test_cloud_pcd_is_read_by_the_reference_s_vendored_pcd_reader(tmp_path, gold):
    """third_party/pypcd.py is the PCD reader the reference ships for its Python tools (run once on these inputs by
    tests/golden/make_golden_keyframe.py): our cloud.pcd is the file it read, and what it read is the cloud."""
    rng = np.random.default_rng(8)
    pts = _cloud(rng, 777)
    d = tmp_path / "kf"; d.mkdir()
    lsdreg.keyframe_save(str(d), 5, 1, pts, np.eye(4))
    assert _sha((d / "cloud.pcd").read_bytes()) == gold["pypcd_pcd_sha256"]
    assert int(gold["pypcd_points"]) == 777 and list(gold["pypcd_fields"]) == ["x", "y", "z", "intensity"]
    assert list(gold["pypcd_sha256"]) == [_sha(pts[:, 0]), _sha(pts[:, 2]), _sha(pts[:, 3] * np.float32(255.0))]
