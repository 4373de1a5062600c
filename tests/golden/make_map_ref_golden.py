#!/usr/bin/env python
"""Record what the reference's own fiducial_slam Map returns (oracle/_ref/libmap_ref.so: map.cpp + transform_with_variance.cpp
compiled unmodified against the stand-in headers of oracle/ref_shim, built by `make -C oracle` where the reference checkout
exists) into tests/golden/map_ref_golden.npz.

tests/test_map_ref.py and tests/test_gpu_slam.py::test_device_map_matches_the_reference_compiled_code compare the numpy
restatement and the CUDA map update with these answers, so they run wherever the repository is checked out.  Every scenario
below feeds the reference exactly the inputs the tests rebuild (seeded synth sequences, the reference test frames of
reference_kat.npz); regenerate when a scenario changes.

Per scenario: <name>_updates rows = published, t[3], q[4] (xyzw), covariance diagonal[6] per Map::update call;
<name>_entries rows = id, x, y, z, roll, pitch, yaw, variance, numObs, n_links (ids ascending);
<name>_links rows = (fiducial, linked fiducial), sorted.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from fiducials_b200 import synth  # noqa: E402
from oracle import map_ref  # noqa: E402
from oracle import slam_oracle as so  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "map_ref_golden.npz")
IDENT7 = [0, 0, 0, 0, 0, 0, 1]
# transform_with_variance operators: every TWV_STRIDE-th of the tests' 2000 seeded random pairs (the special cases at
# it % 7, 11, 13 == 0 all recur in the sample)
TWV_PAIRS, TWV_STRIDE = 2000, 10


def seed_text(se, fmt="%d %f %f %f %f %f %f %f %d\n"):
    return fmt % (*se[:8], 0)


def camera_offset(T_bc):
    inv = so.TWV.from_qt(list(T_bc[3:7]), list(T_bc[0:3]), 0.0).inverse()
    return [*inv.t, *so.m_to_q(inv.R)]


def rand_twv(rng, spread=2.0):
    q = rng.normal(size=4)
    q /= np.linalg.norm(q)
    return [*rng.uniform(-spread, spread, 3), *q, float(10 ** rng.uniform(-6, 2))]


def twv_pairs():
    """The (a, b) pairs of test_transform_with_variance_operators_match_the_reference_code, all TWV_PAIRS of them."""
    rng = np.random.default_rng(0)
    for it in range(TWV_PAIRS):
        a, b = rand_twv(rng), rand_twv(rng)
        if it % 7 == 0:
            b[3:7] = a[3:7]  # identical rotation
        if it % 11 == 0:
            b[3:7] = [-x for x in b[3:7]]  # same rotation, other sign
        if it % 13 == 0:
            b[0:3] = a[0:3]  # identical position: zero-length line between the means
        yield it, a, b


def bag_transforms(kat):
    out = []
    for j, fid in enumerate(kat["bag_golden_ids"].tolist()):
        ge = kat["bag_golden_errs"][j]
        out.append(dict(fiducial_id=fid, translation=kat["bag_golden_t"][j], rotation=kat["bag_golden_q"][j], image_error=ge[0], object_error=ge[1], fiducial_area=ge[2]))
    return out


def img403_fields(kat):
    import cv2

    from oracle import aruco_oracle as ao

    K, D = kat["img403_K"], kat["img403_D"]
    return ao.detect_and_pose(cv2.imdecode(kat["img403_png"], cv2.IMREAD_COLOR), 7, K, D, 0.145)[4]


# auto_init_403.test:3-4: base_link -> camera
IMG403_T_BC = [0.035, 0.145, 0.14, *so.q_from_rpy(-1.204205, -0.041544, -1.479119)]


class Recorder:
    def __init__(self):
        self.out = {}

    def map(self, name, ref):
        self.out[name + "_entries"] = ref.entries()
        self.out[name + "_links"] = np.array(sorted((a, b) for a, bs in ref.links().items() for b in bs), np.int32).reshape(-1, 2)

    def updates(self, name, rows):
        self.out[name + "_updates"] = np.array([[float(pub), *t, *q, *cov] for pub, t, q, cov in rows], np.float64).reshape(-1, 14)


def record_map_ref(rec, kat):
    """The scenarios of tests/test_map_ref.py."""
    for seed in (0, 1, 2):  # test_sequence_with_loaded_origin
        msgs, se = synth.make_c5_sequence(60, seed=seed)
        T_bc = [0.1, -0.02, 0.3, *so.q_from_rpy(0.02, -0.6, 0.1)]
        ref = map_ref.RefMap(initial_map_text=seed_text(se))
        rec.map("seq%d_init" % seed, ref)
        rows = []
        for k, msg in enumerate(msgs):
            rows.append(ref.update(msg, T_bc, camera_offset(T_bc)))
            if k % 10 == 9:
                rec.map("seq%d_k%d" % (seed, k), ref)
        rec.updates("seq%d" % seed, rows)
        ref.close()

    msgs, _ = synth.make_c5_sequence(40, seed=5)  # test_auto_init_then_mapping_and_failed_tf
    ref = map_ref.RefMap()
    T_bc = [0.0, 0.0, 0.2, *so.q_from_rpy(0.0, -0.5, 0.0)]
    rows, states = [], []
    for k, msg in enumerate(msgs):
        lost = k in (17, 18)
        rows.append(ref.update(msg, None if lost else T_bc, None if lost else camera_offset(T_bc)))
        st = ref.state()
        states.append([st["frameNum"], st["isInitializingMap"], st["originFid"]])
    rec.updates("autoinit", rows)
    rec.out["autoinit_state"] = np.array(states, np.int32)
    rec.map("autoinit", ref)
    ref.close()

    msgs, se = synth.make_c5_sequence(30, seed=7)  # test_add_fiducial_clear_and_read_only
    seen = sorted({t["fiducial_id"] for msg in msgs[:12] for t in msg})
    target = [f for f in seen if f != se[0]][0]
    for read_only in (False, True):
        ref = map_ref.RefMap(initial_map_text=seed_text(se), read_only=read_only)
        to_add = []
        for k, msg in enumerate(msgs):
            if k == 3:
                ref.add_fiducial(target)
            T_mb = [0.5, -0.25, 0.0, *so.q_from_rpy(0, 0, 0.3)] if k < 8 else None
            ref.update(msg, IDENT7, IDENT7, T_mapBase=T_mb)
            if k == 20 and not read_only:
                ref.clear()
            to_add.append(ref.state()["fiducialToAdd"])
        rec.out["addfid_ro%d_fiducial_to_add" % read_only] = np.array(to_add, np.int32)
        rec.map("addfid_ro%d" % read_only, ref)
        ref.close()

    msgs, se = synth.make_c5_sequence(12, seed=3)  # test_published_pose_covariance_override_odom_and_squash
    T_ob = [1.0, 2.0, 0.1, *so.q_from_rpy(0.01, -0.02, 0.7)]
    for six_dof in (False, True):
        ref = map_ref.RefMap(initial_map_text=seed_text(se), covariance_diagonal=[0.1, 0.2, 0.3, 0.4, 0.5, 0.6], odom=True, publish_6dof_pose=six_dof)
        rows, tfs = [], []
        for msg in msgs:
            rows.append(ref.update(msg, IDENT7, IDENT7, T_odomBase=T_ob))
            have, tt, tq, is_odom = ref.pose_tf()
            tfs.append([float(have), *tt, *tq, float(is_odom)])
        rec.updates("published_6dof%d" % six_dof, rows)
        rec.out["published_6dof%d_pose_tf" % six_dof] = np.array(tfs, np.float64)
        ref.close()

    msgs, _ = synth.make_c5_sequence(25, seed=9)  # test_map_file_round_trip_through_the_reference
    ref = map_ref.RefMap()
    for msg in msgs:
        ref.update(msg, IDENT7, IDENT7)
    path = os.path.join(ref._dir.name, "saved.txt")
    assert ref.save_map(path)
    text = open(path).read()
    rec.out["roundtrip_saved_map"] = np.frombuffer(text.encode(), np.uint8)
    ref.close()
    ref = map_ref.RefMap(initial_map_text=text)
    rec.map("roundtrip_reloaded", ref)
    ref.close()

    fields = img403_fields(kat)  # test_auto_init_403_golden
    ref = map_ref.RefMap()
    rec.updates("img403", [ref.update(fields, IMG403_T_BC, camera_offset(IMG403_T_BC)) for _ in range(14)])
    rec.map("img403", ref)
    ref.close()

    ref = map_ref.RefMap(initial_map_text="111 0 0 0 0 0 0 0 0\n")  # test_create_map_expectations
    tr = bag_transforms(kat)
    rec.updates("createmap", [ref.update(tr, IDENT7, IDENT7) for _ in range(40)])
    rec.map("createmap", ref)
    ref.close()

    sample = [(it, a, b) for it, a, b in twv_pairs() if it % TWV_STRIDE == 0]  # test_transform_with_variance_operators
    rec.out["twv_index"] = np.array([it for it, _, _ in sample], np.int32)
    for op in ("update", "average", "mul"):
        rec.out["twv_" + op] = np.array([map_ref.twv_apply(op, a, b) for _, a, b in sample])
    rec.out["twv_inverse"] = np.array([map_ref.twv_apply("inverse", a) for _, a, _ in sample])

    def tv(x, var, yaw=0.0):  # test_reference_property_tests_through_the_compiled_reference
        return [x, 0, 0, *so.q_from_rpy(0, 0, yaw), var]

    rec.out["prop_simple"] = map_ref.twv_apply("update", tv(0.0, 1.0), tv(1.0, 1.0))
    rec.out["prop_rotation"] = map_ref.twv_apply("update", tv(0.0, 1.0, 0.0), tv(0.0, 1.0, 1.0))
    cur, it = tv(1.0, 1.0), []
    for _ in range(10):
        cur = map_ref.twv_apply("update", cur, tv(1.0, 1.0)).tolist()
        it.append(cur)
    rec.out["prop_iterated"] = np.array(it)
    rec.out["prop_outlier"] = map_ref.twv_apply("update", tv(0.0, 0.01), tv(10.0, 100.0))
    rec.out["prop_similar"] = map_ref.twv_apply("update", tv(0.0, 1.0), tv(1.0, 1.2))
    # test_zero_variance_observation_gives_nan_like_the_reference
    rec.out["zero_variance"] = map_ref.twv_apply("update", [0, 0, 0, 0, 0, 0, 1, 1.0], [1, 0, 0, 0, 0, 0, 1, 0.0])


def record_c5(rec):
    """test_gpu_slam.py::test_device_map_matches_the_reference_compiled_code: the C5 sequence message by message with a
    camera offset (first 120 messages), and the whole sequence replayed with identity transforms."""
    msgs, se = synth.make_c5_sequence(1000, seed=0)
    text = seed_text(se, "%d %.17g %.17g %.17g %.17g %.17g %.17g %.17g %d\n")
    T_bc = [0.1, -0.02, 0.3, *so.q_from_rpy(0.02, -0.6, 0.1)]
    ref = map_ref.RefMap(initial_map_text=text)
    rec.updates("c5", [ref.update(m, T_bc, camera_offset(T_bc)) for m in msgs[:120]])
    rec.map("c5_k119", ref)
    ref.close()
    ref = map_ref.RefMap(initial_map_text=text)
    ref.replay(msgs, IDENT7, IDENT7)
    rec.out["c5_replay_entries"] = ref.entries()
    ref.close()


def main():
    if not map_ref.available():
        raise SystemExit("%s not built: run `make -C oracle` where the reference checkout exists" % map_ref.LIB_PATH)
    kat = np.load(os.path.join(ROOT, "tests", "golden", "reference_kat.npz"))
    rec = Recorder()
    record_map_ref(rec, kat)
    record_c5(rec)
    np.savez_compressed(OUT, **rec.out)
    print("%s: %d arrays, %d bytes" % (OUT, len(rec.out), os.path.getsize(OUT)))


if __name__ == "__main__":
    main()
