"""oracle/slam_oracle.py (the numpy restatement every map parity test uses) against the REFERENCE'S OWN Map class: fiducial_slam's
map.cpp + transform_with_variance.cpp compiled unmodified from the reference checkout against stand-in ROS / tf2 headers
(oracle/ref_shim, oracle/Makefile -> oracle/_ref/libmap_ref.so).  Same observations in, same map out, to rounding.

What the compiled reference returned for each scenario below is stored in tests/golden/map_ref_golden.npz
(tests/golden/make_map_ref_golden.py feeds it the same inputs), so these tests need no reference checkout."""
import math
import os

import numpy as np
import pytest

from oracle import slam_oracle as so

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = np.load(os.path.join(ROOT, "tests", "golden", "map_ref_golden.npz"))
IDENT7 = [0, 0, 0, 0, 0, 0, 1]


def ref_map(name):
    """(entries, links) of the reference's map at checkpoint `name`: entry rows id, x, y, z, rx, ry, rz, variance, numObs,
    n_links; links {fiducial: set of linked fiducials}."""
    links = {}
    for a, b in GOLDEN[name + "_links"]:
        links.setdefault(int(a), set()).add(int(b))
    return GOLDEN[name + "_entries"], links


def ref_updates(name):
    """The reference's answer to each Map::update call: (published, t3, q4, covariance diagonal)."""
    return [(bool(r[0]), r[1:4], r[4:8], r[8:14]) for r in GOLDEN[name + "_updates"]]


def twv7(t7):
    return so.TWV.from_qt(list(t7[3:7]), list(t7[0:3]), 0.0)


def compare_maps(ref, m: "so.Map", tol=1e-9):
    re, links = ref
    oe = m.entries()
    assert [int(r[0]) for r in re] == [e[0] for e in oe]
    for r, e in zip(re, oe):
        assert np.allclose(r[1:4], e[1:4], rtol=0, atol=tol), (r, e)
        for a, b in zip(r[4:7], e[4:7]):
            d = (a - b + math.pi) % (2 * math.pi) - math.pi
            assert abs(d) < tol, (r, e)
        f = m.fiducials[e[0]]
        assert abs(r[7] - f.pose.var) <= tol * max(1.0, abs(r[7])), (r[7], f.pose.var)
        assert int(r[8]) == f.numObs
    for fid, f in m.fiducials.items():
        assert links.get(fid, set()) == set(f.links), fid


def random_sequence(seed, n_frames=60, n_fids=14):
    """A camera wandering under a ceiling of fiducials, noisy observations (the structure of synth.make_c5_sequence, small)."""
    from fiducials_b200 import synth

    msgs, seed_entry = synth.make_c5_sequence(n_frames, seed=seed)
    return msgs, seed_entry


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_sequence_with_loaded_origin(seed):
    msgs, se = random_sequence(seed)
    T_bc = [0.1, -0.02, 0.3, *so.q_from_rpy(0.02, -0.6, 0.1)]
    inv = twv7(T_bc).inverse()
    T_cb = [*inv.t, *so.m_to_q(inv.R)]
    text = "%d %f %f %f %f %f %f %f %d\n" % (se[0], se[1], se[2], se[3], se[4], se[5], se[6], se[7], 0)
    m = so.Map()
    so.load_map_text(m, text)
    compare_maps(ref_map("seq%d_init" % seed), m)
    updates = ref_updates("seq%d" % seed)
    assert len(updates) == len(msgs)
    for k, msg in enumerate(msgs):
        pub, t, q, cov = updates[k]
        robot = m.update(so.observations_from_transforms(msg), twv7(T_bc), twv7(T_cb))
        assert pub == (robot is not None)
        if pub:
            assert np.allclose(t, robot.t, atol=1e-9)
            qq = so.m_to_q(robot.R)
            assert min(np.abs(np.array(q) - qq).max(), np.abs(np.array(q) + qq).max()) < 1e-9
            assert np.allclose(cov, np.asarray(so.pose_covariance(robot.var)).reshape(6, 6).diagonal(), rtol=1e-12)
        if k % 10 == 9:
            compare_maps(ref_map("seq%d_k%d" % (seed, k)), m)
    assert len(m.fiducials) > 5


def test_auto_init_then_mapping_and_failed_tf():
    msgs, _ = random_sequence(5, n_frames=40)
    updates, states = ref_updates("autoinit"), GOLDEN["autoinit_state"]
    assert len(updates) == len(states) == len(msgs)
    m = so.Map()
    T_bc = [0.0, 0.0, 0.2, *so.q_from_rpy(0.0, -0.5, 0.0)]
    inv = twv7(T_bc).inverse()
    T_cb = [*inv.t, *so.m_to_q(inv.R)]
    for k, msg in enumerate(msgs):
        lost = k in (17, 18)  # the tf look-ups fail for two frames: no pose, no map update (map.cpp:262-272)
        robot = m.update(so.observations_from_transforms(msg), None if lost else twv7(T_bc), None if lost else twv7(T_cb))
        assert updates[k][0] == (robot is not None)
        frame_num, initializing, origin = states[k].tolist()
        assert (frame_num, bool(initializing), origin) == (m.frameNum, m.isInitializingMap, m.originFid)
    compare_maps(ref_map("autoinit"), m)


def test_add_fiducial_clear_and_read_only():
    msgs, se = random_sequence(7, n_frames=30)
    text = "%d %f %f %f %f %f %f %f %d\n" % (se[0], se[1], se[2], se[3], se[4], se[5], se[6], se[7], 0)
    T_bc = IDENT7
    for read_only in (False, True):
        to_add = GOLDEN["addfid_ro%d_fiducial_to_add" % read_only]
        assert len(to_add) == len(msgs)
        m = so.Map(read_only=read_only)
        so.load_map_text(m, text)
        seen = sorted({t["fiducial_id"] for msg in msgs[:12] for t in msg})
        target = [f for f in seen if f != se[0]][0]
        for k, msg in enumerate(msgs):
            if k == 3:
                m.fiducialToAdd = target
            T_mb = [0.5, -0.25, 0.0, *so.q_from_rpy(0, 0, 0.3)] if k < 8 else None  # tf map -> base known early on only
            m.addMapBase = twv7(T_mb) if T_mb is not None else None
            m.update(so.observations_from_transforms(msg), twv7(T_bc), twv7(T_bc))
            if k == 20 and not read_only:
                m.fiducials.clear()  # clearCallback, map.cpp:809-818
                m.initialFrameNum = m.frameNum
                m.originFid = -1
            assert to_add[k] == m.fiducialToAdd
        compare_maps(ref_map("addfid_ro%d" % read_only), m)


def test_published_pose_covariance_override_odom_and_squash():
    msgs, se = random_sequence(3, n_frames=12)
    text = "%d %f %f %f %f %f %f %f %d\n" % (se[0], se[1], se[2], se[3], se[4], se[5], se[6], se[7], 0)
    diag = [0.1, 0.2, 0.3, 0.4, 0.5, 0.6]
    T_ob = [1.0, 2.0, 0.1, *so.q_from_rpy(0.01, -0.02, 0.7)]
    for six_dof in (False, True):
        updates, pose_tfs = ref_updates("published_6dof%d" % six_dof), GOLDEN["published_6dof%d_pose_tf" % six_dof]
        assert len(updates) == len(pose_tfs) == len(msgs)
        m = so.Map()
        so.load_map_text(m, text)
        for k, msg in enumerate(msgs):
            pub, t, q, cov = updates[k]
            robot = m.update(so.observations_from_transforms(msg), so.TWV.identity(), so.TWV.identity())
            assert pub == (robot is not None)
            if pub:
                assert np.allclose(cov, np.asarray(so.pose_covariance(robot.var, diag)).reshape(6, 6).diagonal())
                have, tt, tq, is_odom = bool(pose_tfs[k][0]), pose_tfs[k][1:4], pose_tfs[k][4:8], bool(pose_tfs[k][8])
                exp = so.published_pose_tf(robot, twv7(T_ob), publish_6dof_pose=six_dof)
                eq = np.array(so.m_to_q(exp.R))
                assert have and is_odom
                assert np.allclose(tt, exp.t, atol=1e-9)
                assert min(np.abs(tq - eq).max(), np.abs(tq + eq).max()) < 1e-9


def test_map_file_round_trip_through_the_reference():
    msgs, se = random_sequence(9, n_frames=25)
    m = so.Map()
    for msg in msgs:
        m.update(so.observations_from_transforms(msg), so.TWV.identity(), so.TWV.identity())
    saved = GOLDEN["roundtrip_saved_map"].tobytes().decode()  # the reference's saveMap after the same sequence
    assert saved == so.save_map_text(m)  # byte for byte: same %lf formatting, same link order
    m2 = so.Map()
    so.load_map_text(m2, saved)
    compare_maps(ref_map("roundtrip_reloaded"), m2, tol=1e-12)  # the reference's loadMap of that file


# ---- the reference's own expectations, through the reference's own code -----------------------------------------------------
def _static_tf7(x, y, z, yaw, pitch, roll):
    return [x, y, z, *so.q_from_rpy(roll, pitch, yaw)]


def _replay_against_reference(name, m, transforms, T_bc, T_cb):
    """Feed the restatement the same message once per recorded reference update; same answers, to rounding."""
    for pub, t, q, cov in ref_updates(name):
        robot = m.update(so.observations_from_transforms(transforms), twv7(T_bc), twv7(T_cb))
        assert pub == (robot is not None)
        if pub:
            assert np.allclose(t, robot.t, rtol=0, atol=1e-9)
            qq = np.array(so.m_to_q(robot.R))
            assert min(np.abs(q - qq).max(), np.abs(q + qq).max()) < 1e-9
    compare_maps(ref_map(name), m)
    return pub, t, q


def test_auto_init_403_golden_with_the_reference_code(kat):
    """fiducial_slam/test/auto_init_403_test.cpp:119-137: detect -> pose (cv2) -> the reference's Map -> its golden numbers (1e-3).
    This pins the stand-in tf2 headers as well: a wrong getRPY / slerp / composition order would miss these."""
    from oracle import aruco_oracle as ao

    K, D = kat["img403_K"], kat["img403_D"]
    ids, corners, rvecs, tvecs, fields = ao.detect_and_pose(kat.frame("img403"), 7, K, D, 0.145)
    T_bc = _static_tf7(0.035, 0.145, 0.14, -1.479119, -0.041544, -1.204205)  # auto_init_403.test:3-4  base_link -> camera
    inv = twv7(T_bc).inverse()
    T_cb = [*inv.t, *so.m_to_q(inv.R)]
    assert len(ref_updates("img403")) == 14
    pub, t, q = _replay_against_reference("img403", so.Map(), fields, T_bc, T_cb)
    assert pub
    assert np.abs(np.array([*t, *q]) - [0, 0, 0, 0, 0, 0, 1]).max() < 1e-3
    e = ref_map("img403")[0][0]
    gold = (403, 0.7611, 0.2505, 0.4028, 1.5751, -0.014, -1.546)
    assert int(e[0]) == 403
    assert np.abs(e[1:7] - gold[1:]).max() < 1e-3


def test_create_map_expectations_with_the_reference_code(kat):
    """fiducial_slam/test/create_map_aruco.xml:26-33 (map_test.py, EPSILON 0.1) from the golden transforms of its bag."""
    transforms = []
    for j, fid in enumerate(kat["bag_golden_ids"].tolist()):
        ge = kat["bag_golden_errs"][j]
        transforms.append(dict(fiducial_id=fid, translation=kat["bag_golden_t"][j], rotation=kat["bag_golden_q"][j], image_error=ge[0], object_error=ge[1], fiducial_area=ge[2]))
    m = so.Map()
    so.load_map_text(m, "111 0 0 0 0 0 0 0 0\n")  # 111_initial_map.txt
    assert len(ref_updates("createmap")) == 40
    pub, t, q = _replay_against_reference("createmap", m, transforms, IDENT7, IDENT7)
    assert pub
    exp_pose = [0.73, 0.11, 1.0, 0.98, -0.01, -0.18, 0.07]
    assert np.abs(np.array([*t, *q]) - exp_pose).max() < 0.1
    expect = {100: (-0.27, 0.82, -1.77), 103: (-1.86, -0.59, -1.04), 106: (0.22, -0.0, -0.0), 107: (0.2, -0.28, -0.0), 110: (0.7, 0.05, 0.0), 111: (0.0, 0.0, 0.0), 112: (0.0, -0.3, 0.0)}
    ents = {int(e[0]): e for e in ref_map("createmap")[0]}
    assert sorted(ents) == sorted(expect)
    for fid, g in expect.items():
        assert np.abs(ents[fid][1:4] - g).max() < 0.1


# ---- the fusion operator itself (a10) ----------------------------------------------------------------------------------------
def _rand_twv(rng, spread=2.0):
    q = rng.normal(size=4)
    q /= np.linalg.norm(q)
    return [*rng.uniform(-spread, spread, 3), *q, float(10 ** rng.uniform(-6, 2))]


def _to_so(v):
    return so.TWV.from_qt(list(v[3:7]), list(v[0:3]), v[7])


def _close(ref8, twv, tol=1e-12):
    assert np.allclose(ref8[:3], twv.t, rtol=0, atol=tol * 10)
    q = np.array(so.m_to_q(twv.R))
    assert min(np.abs(ref8[3:7] - q).max(), np.abs(ref8[3:7] + q).max()) < 1e-9
    assert abs(ref8[7] - twv.var) <= 1e-12 * max(1.0, abs(ref8[7]))


def test_transform_with_variance_operators_match_the_reference_code():
    """TransformWithVariance::update / averageTransforms / operator* / inverse of the compiled reference against the restatement the
    whole map oracle is built from, on every tenth of 2000 seeded random pairs (the sample the golden file keeps), incl. equal
    rotations (slerp's theta == 0 branch) and opposite quaternion signs."""
    ref = {op: dict(zip(GOLDEN["twv_index"].tolist(), GOLDEN["twv_" + op])) for op in ("update", "average", "mul", "inverse")}
    assert len(ref["update"]) == 200
    rng = np.random.default_rng(0)
    for it in range(2000):
        a, b = _rand_twv(rng), _rand_twv(rng)
        if it % 7 == 0:
            b[3:7] = a[3:7]  # identical rotation
        if it % 11 == 0:
            b[3:7] = [-x for x in b[3:7]]  # same rotation, other sign
        if it % 13 == 0:
            b[0:3] = a[0:3]  # identical position: zero-length line between the means
        if it not in ref["update"]:
            continue
        A, B = _to_so(a), _to_so(b)
        u = A.copy()
        u.update(B)
        _close(ref["update"][it], u)
        _close(ref["average"][it], so.average_transforms(A, B))
        _close(ref["mul"][it], A.mul(B))
        inv = A.inverse()
        inv.var = A.var
        _close(ref["inverse"][it], inv)


def test_reference_property_tests_through_the_compiled_reference():
    """fiducial_slam/test/transform_var_test.cpp (five inequalities) evaluated with the reference's own operator; the restatement
    gives the same results."""
    def tv(x, var, yaw=0.0):
        return [x, 0, 0, *so.q_from_rpy(0, 0, yaw), var]

    def update(name, a, b):
        u = _to_so(a)
        u.update(_to_so(b))
        r = GOLDEN[name]
        _close(r, u)
        return r

    def angle(v):
        return 2.0 * math.acos(max(-1.0, min(1.0, abs(v[6]))))

    # simple fusion: equal variances meet in the middle, variance shrinks (:15-31)
    r = update("prop_simple", tv(0.0, 1.0), tv(1.0, 1.0))
    assert abs(r[0] - 0.5) < 1e-12 and r[7] < 1.0
    # simple rotation fusion (:33-49)
    r = update("prop_rotation", tv(0.0, 1.0, 0.0), tv(0.0, 1.0, 1.0))
    assert abs(angle(r) - 0.5) < 1e-9
    # same fusion iterated: the estimate stays, the variance falls monotonically (:51-77)
    cur, last = tv(1.0, 1.0), 1.0
    assert len(GOLDEN["prop_iterated"]) == 10
    for r in GOLDEN["prop_iterated"]:
        u = _to_so(cur)
        u.update(_to_so(tv(1.0, 1.0)))
        _close(r, u)
        cur = r.tolist()
        assert abs(cur[0] - 1.0) < 1e-12 and cur[7] <= last
        last = cur[7]
    # an outlier with a large variance barely moves the estimate (:79-107)
    r = update("prop_outlier", tv(0.0, 0.01), tv(10.0, 100.0))
    assert abs(r[0]) < 0.01
    # different estimates with similar variance end up between them (:109-126)
    r = update("prop_similar", tv(0.0, 1.0), tv(1.0, 1.2))
    assert 0.4 < r[0] < 0.6


def test_zero_variance_observation_gives_nan_like_the_reference():
    """object_error == 0 exactly: the reference divides by zero inside probabiltyAtPoint and publishes a NaN variance
    (std::min / std::max let NaN through).  The restatement follows it.  (The device code clamps that NaN to the 1e3 bound --
    slam.cuh normalize_david -- a deliberate difference in a case the detector cannot produce: a reprojection error of exactly 0.)"""
    a = [0, 0, 0, 0, 0, 0, 1, 1.0]
    b = [1, 0, 0, 0, 0, 0, 1, 0.0]
    r = GOLDEN["zero_variance"]
    A = _to_so(a)
    A.update(_to_so(b))
    assert math.isnan(r[7]) and math.isnan(A.var)
    assert np.allclose(r[:3], A.t)
