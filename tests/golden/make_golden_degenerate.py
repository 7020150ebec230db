"""Generates tests/golden/degenerate_ref.npz: laserMapping.cpp compiled unmodified (oracle/_ref/libref_fastlio.so,
RefFastLioBench) on the ground-plane scene of tests/test_oracle_degenerate.py.  Run where oracle/_ref exists:

    python tests/golden/make_golden_degenerate.py

Contents: x (posterior state vector), P (posterior covariance), n_down, n_eff, degenerate.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

import scenes  # noqa: E402
from oracle import eskf  # noqa: E402
from oracle import fastlio as FL  # noqa: E402

assert FL.HAVE_REF_FASTLIO, "oracle/_ref/libref_fastlio.so missing: run `make -C oracle ref` where the reference tree exists"
w = scenes.plane_world()
prior = eskf.State(); prior.rot = eskf.R_to_quat(w["Rprior"]); prior.pos = w["tprior"].copy()
ref = FL.RefFastLioBench(capacity=1 << 30, threads=8)
ref.add_map_points(w["map"])
xr, Pr, n = ref.process_scan(w["scan"], prior, eskf.init_P())
c = ref.counts()
path = os.path.join(HERE, "degenerate_ref.npz")
np.savez_compressed(path, x=xr.to_vec(), P=Pr, n_down=n, n_eff=c["n_eff"], degenerate=c["degenerate"])
print("wrote", path, os.path.getsize(path), "bytes")
