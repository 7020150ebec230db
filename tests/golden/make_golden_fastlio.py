"""Generates tests/golden/fastlio_ref.npz: what the reference's whole LIO front-end (laserMapping.cpp + preprocess.cpp +
ImuProcess + IKFoM + iVox compiled unmodified into oracle/_ref/libref_fastlio.so by oracle/Makefile) answers, frame by
frame, on the synthetic sensor stream of tests/test_oracle_fastlio.py.  Run where oracle/_ref exists:

    python tests/golden/make_golden_fastlio.py

Contents, per extrinsic (prefix `ext` / `noext`), one row per frame of the 17-frame stream:
  {p}_step, {p}_init      fastlio_main's return value and ImuProcess::IsInit after the frame
  {p}_counts              n_down, n_eff, map_cells, degenerate
  {p}_x, {p}_P            the posterior state vector and covariance
  {p}_down_sha256         sha256 of the downsampled cloud (float32 [n,4])
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

import test_oracle_fastlio as T  # noqa: E402  (the tests' own stream)
from oracle import fastlio as F  # noqa: E402

assert F.HAVE_REF_FASTLIO, "oracle/_ref/libref_fastlio.so missing: run `make -C oracle ref` where the reference tree exists"

out = {}
for ext in (False, True):
    p = "ext" if ext else "noext"
    ext_R, ext_t = T._extrinsic(ext)
    ref = F.RefFastLio(ext_R, ext_t)
    rows = dict(step=[], init=[], counts=[], x=[], P=[], down_sha256=[])
    for frame in T._stream(17, ext_R, ext_t):
        T._feed(ref, *frame)
        rows["step"].append(ref.step())
        rows["init"].append(ref.initialised)
        c = ref.counts()
        rows["counts"].append([c["n_down"], c["n_eff"], c["map_cells"], c["degenerate"]])
        x, P = ref.state()
        rows["x"].append(x.to_vec()); rows["P"].append(P)
        rows["down_sha256"].append(hashlib.sha256(np.ascontiguousarray(ref.downsampled(), np.float32).tobytes()).hexdigest())
    for k, v in rows.items():
        out[f"{p}_{k}"] = np.array(v)
path = os.path.join(HERE, "fastlio_ref.npz")
np.savez_compressed(path, **out)
print("wrote", path, os.path.getsize(path), "bytes")
