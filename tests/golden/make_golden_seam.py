"""Generates tests/golden/seam_ref.npz: what the reference's front-end (oracle/_ref/libref_fastlio.so, filter_num 3,
undistortion off) downsamples, frame by frame, from the stream of tests/test_fastlio_seam_host.py's decimation test.
Run where oracle/_ref exists:

    python tests/golden/make_golden_seam.py

Contents, one row per frame: step (fastlio_main's return value), n_down, down_xyz_sha256 (sha256 of the float32 x, y, z
columns of the downsampled cloud, C order).
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

import test_oracle_fastlio as T  # noqa: E402  (the stream the seam test feeds)
from oracle import fastlio as F  # noqa: E402

assert F.HAVE_REF_FASTLIO, "oracle/_ref/libref_fastlio.so missing: run `make -C oracle ref` where the reference tree exists"
ext_R, ext_t = np.eye(3), np.zeros(3)
ref = F.RefFastLio(ext_R, ext_t, filter_num=3, undistort=False)
step, n_down, sha = [], [], []
for fr in T._stream(8, ext_R, ext_t, n_az=120):
    T._feed(ref, *fr)
    step.append(ref.step())
    n_down.append(ref.counts()["n_down"])
    sha.append(hashlib.sha256(np.ascontiguousarray(ref.downsampled()[:, :3], np.float32).tobytes()).hexdigest())
path = os.path.join(HERE, "seam_ref.npz")
np.savez_compressed(path, step=np.array(step), n_down=np.array(n_down), down_xyz_sha256=np.array(sha))
print("wrote", path, os.path.getsize(path), "bytes")
