"""ctypes front end of oracle/_ref/libmap_ref.so: the REFERENCE's own fiducial_slam Map (map.cpp + transform_with_variance.cpp compiled
unmodified from /root/reference against the stand-in headers of oracle/ref_shim; built by oracle/Makefile where the reference
checkout exists, shipped prebuilt to the GPU box).

TEST INFRASTRUCTURE ONLY -- never imported by the product (fiducials_b200/).  tests/golden/make_map_ref_golden.py records its answers
into tests/golden/map_ref_golden.npz, against which tests/test_map_ref.py pins oracle/slam_oracle.py and tests/test_gpu_slam.py
checks the CUDA map update: the reference code itself rather than a restatement, without needing the reference checkout."""
import ctypes as C
import os
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_ref", "libmap_ref.so")
_lib = None


def available() -> bool:
    return os.path.exists(LIB_PATH)


def _load():
    global _lib
    if _lib is None:
        lib = C.CDLL(LIB_PATH)
        lib.mapref_create.restype = C.c_void_p
        lib.mapref_create.argtypes = [C.c_double, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_char_p, C.c_char_p, C.c_char_p]
        lib.mapref_destroy.argtypes = [C.c_void_p]
        lib.mapref_set_tf.argtypes = [C.c_char_p, C.c_char_p, C.c_void_p]
        lib.mapref_update.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_char_p, C.c_void_p]
        lib.mapref_entries.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        lib.mapref_links.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        lib.mapref_pose_tf.argtypes = [C.c_void_p, C.c_void_p]
        lib.mapref_add_fiducial.argtypes = [C.c_void_p, C.c_int]
        lib.mapref_clear.argtypes = [C.c_void_p]
        lib.mapref_load_map.argtypes = [C.c_void_p, C.c_char_p]
        lib.mapref_save_map.argtypes = [C.c_void_p, C.c_char_p]
        lib.mapref_state.argtypes = [C.c_void_p, C.c_void_p]
        lib.twvref_apply.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.mapref_replay.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_char_p]
        _lib = lib
    return _lib


def twv_apply(op, a, b=None):
    """The reference's TransformWithVariance, directly.  a, b: x y z qx qy qz qw variance.  op: 'update', 'average', 'mul', 'inverse'."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b if b is not None else a, np.float64)
    out = np.zeros(8, np.float64)
    _load().twvref_apply({"update": 0, "average": 1, "mul": 2, "inverse": 3}[op], a.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
    return out


CAMERA, BASE, MAP, ODOM = b"camera", b"base_link", b"map", b"odom"


class RefMap:
    """One Map instance of the reference.  tf look-ups are process-global in the stand-in buffer: set_tf before every update."""

    def __init__(self, weighting_scale=1e9, use_area=False, read_only=False, publish_6dof_pose=False, covariance_diagonal=None, odom=False, initial_map_text=None):
        lib = _load()
        self._dir = tempfile.TemporaryDirectory()
        self.map_file = os.path.join(self._dir.name, "map.txt")
        if initial_map_text is not None:
            with open(self.map_file, "w") as f:
                f.write(initial_map_text)
        cov = np.asarray(covariance_diagonal, np.float64) if covariance_diagonal is not None else None
        lib.mapref_clear_tf()
        self.h = C.c_void_p(lib.mapref_create(float(weighting_scale), int(use_area), int(read_only), int(publish_6dof_pose), cov.ctypes.data_as(C.c_void_p) if cov is not None else None,
                                              self.map_file.encode(), ODOM if odom else b"", BASE))
        self.stamp = 100.0

    def close(self):
        if self.h:
            _load().mapref_destroy(self.h)
            self.h = None
            self._dir.cleanup()

    @staticmethod
    def set_tf(target: bytes, source: bytes, t7):
        """t7 = x y z qx qy qz qw, the answer of lookupTransform(target, source); None removes nothing (clear_tf() resets all)."""
        a = np.asarray(t7, np.float64)
        _load().mapref_set_tf(target, source, a.ctypes.data_as(C.c_void_p))

    @staticmethod
    def clear_tf():
        _load().mapref_clear_tf()

    def update(self, transforms, T_baseCam=None, T_camBase=None, T_mapBase=None, T_odomBase=None):
        """transforms: dicts with fiducial_id, translation, rotation (xyzw), object_error, fiducial_area.  T_*: 7-vectors or None
        (= that tf look-up fails).  Returns (published, t3, q4, covariance diagonal)."""
        self.clear_tf()
        if T_baseCam is not None:
            self.set_tf(BASE, CAMERA, T_baseCam)
        if T_camBase is not None:
            self.set_tf(CAMERA, BASE, T_camBase)
        if T_mapBase is not None:
            self.set_tf(MAP, BASE, T_mapBase)
        if T_odomBase is not None:
            self.set_tf(ODOM, BASE, T_odomBase)
        obs = np.zeros((len(transforms), 10), np.float64)
        for i, t in enumerate(transforms):
            obs[i] = [t["fiducial_id"], *t["translation"], *t["rotation"], t["object_error"], t["fiducial_area"]]
        out = np.zeros(14, np.float64)
        self.stamp += 0.05
        _load().mapref_update(self.h, len(transforms), obs.ctypes.data_as(C.c_void_p), self.stamp, CAMERA, out.ctypes.data_as(C.c_void_p))
        return bool(out[0]), out[1:4].copy(), out[4:8].copy(), out[8:14].copy()

    def replay(self, messages, T_baseCam=None, T_camBase=None):
        """The whole message sequence inside the compiled reference (one call; used for timing).  Returns the number of fiducials."""
        self.clear_tf()
        if T_baseCam is not None:
            self.set_tf(BASE, CAMERA, T_baseCam)
        if T_camBase is not None:
            self.set_tf(CAMERA, BASE, T_camBase)
        flat = np.array([[t["fiducial_id"], *t["translation"], *t["rotation"], t["object_error"], t["fiducial_area"]] for msg in messages for t in msg], np.float64).reshape(-1, 10)
        off = np.zeros(len(messages) + 1, np.int32)
        off[1:] = np.cumsum([len(m) for m in messages])
        self._replay_args = (flat, off)
        return _load().mapref_replay(self.h, len(messages), off.ctypes.data_as(C.c_void_p), flat.ctypes.data_as(C.c_void_p), self.stamp, CAMERA)

    def entries(self):
        """rows: id, x, y, z, rx, ry, rz, variance, numObs, n_links (ids ascending)"""
        out = np.zeros((4096, 10), np.float64)
        n = _load().mapref_entries(self.h, 4096, out.ctypes.data_as(C.c_void_p))
        return out[:n].copy()

    def links(self):
        buf = np.zeros((65536, 2), np.int32)
        n = _load().mapref_links(self.h, 65536, buf.ctypes.data_as(C.c_void_p))
        d = {}
        for a, b in buf[:n]:
            d.setdefault(int(a), set()).add(int(b))
        return d

    def pose_tf(self):
        out = np.zeros(9, np.float64)
        _load().mapref_pose_tf(self.h, out.ctypes.data_as(C.c_void_p))
        return bool(out[0]), out[1:4].copy(), out[4:8].copy(), bool(out[8])

    def add_fiducial(self, fid):
        _load().mapref_add_fiducial(self.h, int(fid))

    def clear(self):
        _load().mapref_clear(self.h)

    def save_map(self, path):
        return bool(_load().mapref_save_map(self.h, path.encode()))

    def load_map(self, path):
        return bool(_load().mapref_load_map(self.h, path.encode()))

    def state(self):
        s = np.zeros(4, np.int32)
        _load().mapref_state(self.h, s.ctypes.data_as(C.c_void_p))
        return dict(frameNum=int(s[0]), isInitializingMap=bool(s[1]), originFid=int(s[2]), fiducialToAdd=int(s[3]))
