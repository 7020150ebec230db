"""Generates tests/golden/keyframe_ref.npz: what the reference's key-frame code (KeyFrame::save / loadOdom / loadPcd compiled
unmodified into oracle/_ref/libref_keyframe.so by oracle/Makefile) and the PCD reader it vendors (third_party/pypcd.py)
produce on the seeded inputs of tests/test_keyframe_io.py.  Run where the reference tree and oracle/_ref exist:

    python tests/golden/make_golden_keyframe.py REFERENCE_TREE      (the original project's checkout)

Contents:
  save{k}_data            bytes of the `data` file KeyFrame::save wrote for key frame k (uint8)
  save_pcd_sha256         sha256 of each cloud.pcd it wrote
  load{k}_data, load{k}_pcd   the files it wrote for the load test's key frames (uint8)
  load_stamp, load_id, load_T, load_n, load_pts_sha256
                          what KeyFrame::loadOdom / loadPcd returned reading those files
  pypcd_pcd_sha256        sha256 of the cloud.pcd pypcd read (KeyFrame::save's, for the pypcd test's inputs)
  pypcd_points, pypcd_fields, pypcd_sha256
                          pypcd.PointCloud.from_path on it: point count, field names, sha256 of x, z, intensity
"""
import ctypes as C
import hashlib
import os
import sys
import tempfile
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

import test_keyframe_io as T  # noqa: E402  (the tests' own input generators)


def _ref():
    L = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_keyframe.so"))
    f = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
    d = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
    L.ref_keyframe_save.argtypes = [C.c_char_p, C.c_uint64, C.c_long, f, C.c_int, d]
    L.ref_keyframe_load.restype = C.c_int
    L.ref_keyframe_load.argtypes = [C.c_char_p, C.POINTER(C.c_uint64), C.POINTER(C.c_long), d, f, C.c_int]
    return L


def sha(b) -> str:
    return hashlib.sha256(b if isinstance(b, bytes) else np.ascontiguousarray(b).tobytes()).hexdigest()


def u8(b: bytes) -> np.ndarray:
    return np.frombuffer(b, np.uint8).copy()


def main(ref_tree: str) -> None:
    L = _ref()
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        rng = np.random.default_rng(4)
        shas = []
        for k, P in enumerate(T._poses(rng)):
            pts = T._cloud(rng, 1000 + 37 * k)
            d = os.path.join(tmp, f"save{k}"); os.mkdir(d)
            L.ref_keyframe_save(os.fsencode(d), 1_695_000_000_000_000 + 123_456 * k + 7, 40 + k, pts, pts.shape[0],
                                np.ascontiguousarray(P, np.float64).reshape(-1))
            out[f"save{k}_data"] = u8(open(os.path.join(d, "data"), "rb").read())
            shas.append(sha(open(os.path.join(d, "cloud.pcd"), "rb").read()))
        out["save_pcd_sha256"] = np.array(shas)

        rng = np.random.default_rng(5)
        stamps, ids, Ts, ns, pshas = [], [], [], [], []
        for k, P in enumerate(T._poses(rng)[:4]):
            pts = T._cloud(rng, 500 + k)
            d = os.path.join(tmp, f"load{k}"); os.mkdir(d)
            L.ref_keyframe_save(os.fsencode(d), 1_700_000_000_000_000 + 999_999 - k, 7 + k, pts, pts.shape[0],
                                np.ascontiguousarray(P, np.float64).reshape(-1))
            out[f"load{k}_data"] = u8(open(os.path.join(d, "data"), "rb").read())
            out[f"load{k}_pcd"] = u8(open(os.path.join(d, "cloud.pcd"), "rb").read())
            s, i = C.c_uint64(), C.c_long()
            T2 = np.zeros(16); p2 = np.zeros((pts.shape[0], 4), np.float32)
            ns.append(L.ref_keyframe_load(os.fsencode(d), C.byref(s), C.byref(i), T2, p2, p2.shape[0]))
            stamps.append(s.value); ids.append(i.value); Ts.append(T2.reshape(4, 4)); pshas.append(sha(p2))
        out.update(load_stamp=np.array(stamps, np.uint64), load_id=np.array(ids, np.int64), load_T=np.array(Ts),
                   load_n=np.array(ns, np.int64), load_pts_sha256=np.array(pshas))

        sys.modules.setdefault("lzf", types.ModuleType("lzf"))
        sys.path.insert(0, os.path.join(ref_tree, "third_party"))
        import pypcd
        rng = np.random.default_rng(8)
        pts = T._cloud(rng, 777)
        d = os.path.join(tmp, "pypcd"); os.mkdir(d)
        L.ref_keyframe_save(os.fsencode(d), 5, 1, pts, pts.shape[0], np.eye(4).reshape(-1))
        f = os.path.join(d, "cloud.pcd")
        out["pypcd_pcd_sha256"] = np.array(sha(open(f, "rb").read()))
        # numpy 2 dropped the binary mode of np.fromstring the reader was written against: route that call to np.frombuffer
        pypcd.np.fromstring = lambda buf, dtype=float, **kw: np.frombuffer(buf, dtype=dtype)
        pc = pypcd.PointCloud.from_path(f)
        out.update(pypcd_points=np.array(pc.points), pypcd_fields=np.array(list(pc.fields)),
                   pypcd_sha256=np.array([sha(pc.pc_data[c]) for c in ("x", "z", "intensity")]))
    path = os.path.join(HERE, "keyframe_ref.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main(sys.argv[1])
