"""CPU: the host side of the LIO seam (csrc/fastlio_seam.cu: queues, Preprocess::velodyne_handler's decimation and blind
zone, sync_packages, the default outputs of fastlio_state / fastlio_odometry) against the restated pipeline
(oracle/fastlio.py::OracleFastLio, pinned to the compiled reference by tests/test_oracle_fastlio.py) and, where
oracle/_ref exists, against what the compiled reference itself consumes.  No device is touched: lsd_fastlio_pop_package
is sync_packages alone.  The product must fail loudly, not fall back, when lsd_fastlio_main needs the GPU."""
import numpy as np
import pytest

import lsdreg
from oracle import fastlio as F

import test_oracle_fastlio as T


def _packages(p, pop):
    out = []
    while True:
        m = pop(p)
        if m is None:
            return out
        out.append(m)


@pytest.mark.parametrize("filter_num,max_point_num", [(1, -1), (3, -1), (1, 5000)])
def test_packages_match_the_restated_sync(filter_num, max_point_num):
    ext_R, ext_t = np.eye(3), np.array([0.1, -0.05, 0.2])
    g = lsdreg.FastLio(ext_R, ext_t, filter_num=filter_num, max_point_num=max_point_num)
    o = F.OracleFastLio(ext_R, ext_t, filter_num=filter_num, max_point_num=max_point_num)
    frames = list(T._stream(6, ext_R, ext_t, n_az=120))
    # a scan with points inside the blind zone and exactly on its border, IMU samples exactly at a scan's end time
    frames[2][1][:50, :3] *= np.float32(0.001)
    frames[2][1][50, :3] = np.array([0.1, 0.0, 0.0], np.float32)
    got, want = [], []
    for k, fr in enumerate(frames):
        T._feed(g, *fr); T._feed(o, *fr)
        if k % 2 == 1:      # two scans queued before the consumer runs: packages must come out in order with the right IMU split
            got += _packages(g, lambda p: p.pop_package())
            want += _packages(o, lambda p: p._sync())
    assert len(got) == len(want) == 6
    for a, b in zip(got, want):
        assert a["lidar_beg_time"] == b["lidar_beg_time"] and a["lidar_end_time"] == b["lidar_end_time"]
        np.testing.assert_array_equal(a["points"], b["points"])
        np.testing.assert_array_equal(a["time_ms"], b["time_ms"])
        np.testing.assert_array_equal(a["imu"], b["imu"])
        assert a["ins_vel"] is None
    assert g.pop_package() is None
    # no scan without IMU, no IMU without scan (sync_packages :448-450)
    g.push_scan(frames[0][1], frames[0][2], 10_000_000)
    assert g.pop_package() is None
    g.push_imu(10.05, np.zeros(3), np.array([0, 0, 1.0]))
    m = g.pop_package()
    assert m is not None and m["imu"].shape == (1, 7) and m["imu"][0, 6] == 1.0 * 9.81 / 9.81


def test_ins_velocity_is_rotated_into_the_imu_frame():
    """fastlio_ins_enqueue (laserMapping.cpp:418-443): ENU -> ego by getTransformFromRPYT(0,0,0,-heading,pitch,roll)^-1, then
    Lidar_R_wrt_IMU; up component dropped; only the last sample before the scan end is used; invalid non-wheel samples ignored."""
    ext_R = lsdreg.synth.rot_from_rpy(0.02, -0.01, 0.3)
    g = lsdreg.FastLio(ext_R, np.zeros(3))
    g.push_ins(20_000, [9.0, 9.0, 9.0], 10.0, 0.0, 0.0, rtk_valid=False, is_wheel=False)       # dropped
    g.push_ins(30_000, [1.0, 2.0, 0.5], 30.0, 2.0, -1.0)
    g.push_ins(60_000, [3.0, -1.0, 0.2], 40.0, 1.0, 3.0, rtk_valid=False, is_wheel=True)
    g.push_ins(160_000, [7.0, 7.0, 7.0], 0.0, 0.0, 0.0)                                         # after the scan end
    g.push_imu(0.05, np.zeros(3), np.array([0, 0, 1.0]))
    g.push_scan(np.array([[5, 0, 0, 1]], np.float32), np.array([0], np.uint32), 0)
    m = g.pop_package()
    k = np.pi / 180.0
    def rot(axis, a):
        c, s = np.cos(a), np.sin(a)
        return {"z": np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]]), "x": np.array([[1, 0, 0], [0, c, -s], [0, s, c]]),
                "y": np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]])}[axis]
    Rve = rot("z", -40.0 * k) @ rot("x", 1.0 * k) @ rot("y", 3.0 * k)
    v = ext_R @ (Rve.T @ np.array([3.0, -1.0, 0.2]))
    np.testing.assert_allclose(m["ins_vel"], [v[0], v[1], 0.0], rtol=0, atol=1e-15)


def test_outputs_before_any_scan_and_loud_failure_without_a_device():
    import torch
    g = lsdreg.FastLio()
    assert not g.initialised
    s, e = g.odometry()
    np.testing.assert_array_equal(s, np.eye(4)); np.testing.assert_array_equal(e, np.eye(4))
    st = g.state()
    np.testing.assert_array_equal(st[:7], [0, 0, 0, 0, 0, 0, 1])
    np.testing.assert_array_equal(st[16:19], [9.809, 0, 0])       # S2(): length * e_x until IMU_init
    assert g.step() is False                                      # nothing queued
    fr = list(T._stream(2, np.eye(3), np.zeros(3), n_az=60))
    T._feed(g, *fr[0]); T._feed(g, *fr[1])
    assert g.step() is True                                       # the first scan only sets first_lidar_time (:1171-1177)
    if not torch.cuda.is_available():
        with pytest.raises(lsdreg.LsdError) as ei:                # the second needs the device: no CPU fallback
            g.step()
        assert ei.value.status == lsdreg.ERR_NO_DEVICE


def test_decimation_matches_what_the_compiled_reference_consumes():
    """The compiled reference, fed the same raw scans through fastlio_pcl_enqueue, downsamples exactly the points this seam
    keeps: its feats_down (VoxelGrid of the undistorted cloud, undistort off) equals the VoxelGrid of our package.  The
    reference's side is its answer on this stream, recorded by tests/golden/make_golden_seam.py."""
    import hashlib
    import os
    from oracle import oracle as O
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "seam_ref.npz"))
    ext_R, ext_t = np.eye(3), np.zeros(3)
    g = lsdreg.FastLio(ext_R, ext_t, filter_num=3, undistort=False)
    seen = 0
    for k, fr in enumerate(T._stream(8, ext_R, ext_t, n_az=120)):
        T._feed(g, *fr)
        assert gold["step"][k]
        m = g.pop_package()
        if gold["n_down"][k] > 0 and k >= 6:
            got = O.voxelgrid(m["points"], 0.5)
            assert got.shape[0] == gold["n_down"][k]
            assert hashlib.sha256(np.ascontiguousarray(got[:, :3], np.float32).tobytes()).hexdigest() == gold["down_xyz_sha256"][k]
            seen += 1
    assert seen >= 1
