"""CPU: the degeneracy branch of h_share_model_geometric (laserMapping.cpp:934-980) pinned against the compiled reference.

Scene: nothing but the ground plane (tests/scenes.py::plane_world) — every plane normal is +-e_z, so two eigen-directions of
the 3x3 normal block fall below the reference's 250 / 50 contribution thresholds and the Jacobian rows are projected
(mat_p, :975-978).  The restated pipeline (oracle/lio.py + lsd_oracle.c) and laserMapping.cpp compiled unmodified
(oracle/_ref/libref_fastlio.so, RefFastLioBench; its answer on this scene is tests/golden/degenerate_ref.npz, recorded by
tests/golden/make_golden_degenerate.py) must flag the same scan as degenerate and end at the same pose.
tests/test_gpu_lio.py::test_degenerate_scene_projection holds the CUDA path to the restated pipeline on the same scene."""
import os

import numpy as np

import scenes
from oracle import eskf
from oracle.lio import OracleLio

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "degenerate_ref.npz")


def test_degenerate_scene_oracle_equals_compiled_reference():
    w = scenes.plane_world()
    prior = eskf.State(); prior.rot = eskf.R_to_quat(w["Rprior"]); prior.pos = w["tprior"].copy()
    o = OracleLio(18, expected_cells=1 << 18, stale_neighbours=True)
    o.add_map_points(w["map"])
    r = o.process_scan(w["scan"], prior, eskf.init_P())
    assert all(l["degenerate"] == 1 for l in r["log"]) and r["log"][-1]["n_eff"] > 3000
    g = np.load(GOLD)
    xr, Pr = eskf.State.from_vec(g["x"].copy()), g["P"]
    assert int(g["degenerate"]) == 1 and int(g["n_eff"]) == r["log"][-1]["n_eff"] and int(g["n_down"]) == r["n_down"]
    d = np.abs(o.x.boxminus(xr))
    assert d[:3].max() < 1e-6 and d[3:6].max() < 1e-7, d[:6]
    np.testing.assert_allclose(o.P, Pr, rtol=1e-5, atol=1e-6)      # unobservable directions: entries of 1e-10 are rounding noise
    # the projection did its job: x / y stay where the prior put them, z is pulled onto the plane
    assert np.abs(o.x.pos[:2] - w["tprior"][:2]).max() < 1e-3 and abs(o.x.pos[2] - w["tgt"][2]) < 5e-3
