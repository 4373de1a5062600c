"""GPU parity of the fiducial_slam update through the C-ABI vs the numpy restatement
(oracle/slam_oracle.py) and the reference's goldens.  Tolerance: map poses within 1e-4 m / 1e-4 rad
(BASELINE.md section 4); in practice ~1e-12."""
import math
import os

import numpy as np
import pytest

from oracle import slam_oracle as so

pytestmark = pytest.mark.gpu


def _bag_transforms(kat):
    out = []
    for j, fid in enumerate(kat["bag_golden_ids"].tolist()):
        ge = kat["bag_golden_errs"][j]
        out.append(dict(fiducial_id=fid, translation=kat["bag_golden_t"][j], rotation=kat["bag_golden_q"][j], image_error=ge[0], object_error=ge[1], fiducial_area=ge[2]))
    return out


def _tf7(T):
    return np.array(T.t + so.m_to_q(T.R))


def _cmp_entries(dev_entries, ref_entries, tol=1e-4):
    assert [e.fiducial_id for e in dev_entries] == [r[0] for r in ref_entries]
    for e, r in zip(dev_entries, ref_entries):
        got = np.array([e.x, e.y, e.z, e.rx, e.ry, e.rz])
        assert np.abs(got - np.array(r[1:7])).max() < tol


def test_create_map_sequence(kat):
    from fiducials_b200.node import FiducialSlam

    tr = _bag_transforms(kat)
    ident = so.TWV.identity()
    ref = so.Map()
    ref.load_entry(111, 0, 0, 0, 0, 0, 0, 0, 0)
    slam = FiducialSlam(max_fiducials=32)
    slam.loadMap([[111, 0, 0, 0, 0, 0, 0, 0, 0]])
    for _ in range(40):
        rr = ref.update(so.observations_from_transforms(tr), ident, ident)
        r = slam.transformCallback(tr, _tf7(ident), _tf7(ident))
        assert r.valid == 1 and np.abs(np.array(r.t) - np.array(rr.t)).max() < 1e-4
    _cmp_entries(slam.entries(), ref.entries(), 1e-9)
    # reference expectations, create_map_aruco.xml:26-33 (EPSILON 0.1)
    ents = {e.fiducial_id: e for e in slam.entries()}
    assert abs(ents[100].x + 0.27) < 0.1 and abs(ents[100].y - 0.82) < 0.1 and abs(ents[100].z + 1.77) < 0.1
    assert abs(math.degrees(ents[103].ry) + 23.72) < 1.0
    msg = slam.publishMap()
    assert [f.fiducial_id for f in msg.fiducials] == sorted(ents)


def test_save_and_load_map_file(kat, tmp_path):
    """saveMap / loadMap (map.cpp:541-625) through the device map: after the create_map sequence the file written
    from the GPU state equals the oracle's line for line (ids, numObs and links exactly, values to the file's %lf
    precision); loading it into a fresh handle and replaying gives the oracle's result for the same history."""
    from fiducials_b200.node import FiducialSlam

    tr = _bag_transforms(kat)
    ident = so.TWV.identity()
    ref = so.Map()
    ref.load_entry(111, 0, 0, 0, 0, 0, 0, 0, 0)
    slam = FiducialSlam(max_fiducials=32)
    slam.loadMap([[111, 0, 0, 0, 0, 0, 0, 0, 0]])
    for _ in range(15):
        ref.update(so.observations_from_transforms(tr), ident, ident)
        slam.transformCallback(tr, _tf7(ident), _tf7(ident))
    path = tmp_path / "map.txt"
    assert slam.saveMap(str(path))
    got = [l.split() for l in path.read_text().splitlines()]
    exp = [l.split() for l in so.save_map_text(ref).splitlines()]
    assert len(got) == len(exp) == len(ref.fiducials) and len(exp) > 3
    for g, e in zip(got, exp):
        assert g[0] == e[0] and g[8:] == e[8:] and len(g) > 9  # id, numObs, links
        assert np.abs(np.array(g[1:8], float) - np.array(e[1:8], float)).max() <= 2e-6
    # load into fresh maps (device and oracle) and keep going: same history -> same result
    slam2 = FiducialSlam(max_fiducials=32)
    assert slam2.loadMapFile(str(path)) == len(exp)
    assert slam2.links() == slam.links()
    ref2 = so.Map()
    so.load_map_text(ref2, path.read_text())
    for _ in range(5):
        ref2.update(so.observations_from_transforms(tr), ident, ident)
        slam2.transformCallback(tr, _tf7(ident), _tf7(ident))
    _cmp_entries(slam2.entries(), ref2.entries(), 1e-9)
    slam.close()
    slam2.close()


def test_auto_init_403_golden(kat):
    from fiducials_b200.node import Detector, FiducialSlam, default_params

    det = Detector(default_params(dictionary=7), 0, 1280, 960, 1)
    ids, corners = det.detect(kat.frame("img403"))
    tfs = det.pose(ids, corners, kat["img403_K"], kat["img403_D"], 0.145)
    det.close()
    fields = [dict(fiducial_id=t.fiducial_id, translation=list(t.translation), rotation=list(t.rotation), image_error=t.image_error, object_error=t.object_error,
                   fiducial_area=t.fiducial_area) for t in tfs]
    T_baseCam = so.TWV.from_qt(so.q_from_rpy(-1.204205, -0.041544, -1.479119), [0.035, 0.145, 0.14])  # auto_init_403.test:3-4
    T_camBase = T_baseCam.inverse()
    slam = FiducialSlam(max_fiducials=8)
    for _ in range(14):
        r = slam.transformCallback(fields, _tf7(T_baseCam), _tf7(T_camBase))
    assert r.valid == 1
    assert np.abs(np.array(r.t)).max() < 1e-3 and abs(r.q[3] - 1) < 1e-3  # auto_init_403_test.cpp:119-126
    e = slam.entries()[0]
    gold = [0.7611, 0.2505, 0.4028, 1.5751, -0.014, -1.546]  # :128-137
    assert e.fiducial_id == 403 and np.abs(np.array([e.x, e.y, e.z, e.rx, e.ry, e.rz]) - np.array(gold)).max() < 1e-3


def _random_walk_messages(rng, n_fid, n_msgs, per_msg):
    """Synthetic C5-style sequence: fiducials on a ceiling grid, camera moving below."""
    grid = [(float(i % 5), float(i // 5), 2.5) for i in range(n_fid)]
    msgs = []
    for k in range(n_msgs):
        cam = np.array([2.0 + 1.5 * math.sin(0.07 * k), 1.0 + 1.0 * math.cos(0.05 * k), 0.0])
        vis = sorted(range(n_fid), key=lambda i: (grid[i][0] - cam[0]) ** 2 + (grid[i][1] - cam[1]) ** 2)[:per_msg]
        rng.shuffle(vis)
        m = []
        for i in vis:
            t = np.array(grid[i]) - cam + rng.normal(0, 0.005, 3)
            q = so.q_from_rpy(math.pi + rng.normal(0, 0.01), rng.normal(0, 0.01), math.pi + rng.normal(0, 0.01))
            m.append(dict(fiducial_id=100 + i, translation=t, rotation=np.array(q), image_error=0.1, object_error=float(rng.uniform(1e-4, 1e-2)), fiducial_area=1000.0))
        msgs.append(m)
    return msgs, grid


def test_replay_sequence_matches_oracle_and_is_order_dependent():
    from fiducials_b200.node import FiducialSlam

    rng = np.random.default_rng(0)
    msgs, grid = _random_walk_messages(rng, 20, 120, 6)
    ident = so.TWV.identity()
    ref = so.Map()
    ref.load_entry(100, grid[0][0], grid[0][1], grid[0][2], 180, 0, 180, 0, 0)
    robots_ref = [ref.update(so.observations_from_transforms(m), ident, ident) for m in msgs]
    slam = FiducialSlam(max_fiducials=64, n_instances=2)
    for inst in range(2):
        slam.loadMap([[100, grid[0][0], grid[0][1], grid[0][2], 180, 0, 180, 0, 0]], instance=inst)
    rev = [list(reversed(m)) for m in msgs]  # instance 1 sees every message in reversed order
    robots = slam.replay([msgs, rev], _tf7(ident), _tf7(ident))
    _cmp_entries(slam.entries(0), ref.entries(), 1e-4)
    _cmp_entries(slam.entries(0), ref.entries(), 1e-9)
    for k, rr in enumerate(robots_ref):
        if rr is not None:
            assert robots[k].valid == 1 and np.abs(np.array(robots[k].t) - np.array(rr.t)).max() < 1e-9
    # the fold is order dependent (SURVEY fact 6): reversed message order gives a (slightly) different map
    a = np.array([[e.x, e.y, e.z] for e in slam.entries(0)])
    b = np.array([[e.x, e.y, e.z] for e in slam.entries(1)])
    assert a.shape == b.shape and np.abs(a - b).max() > 0 and np.abs(a - b).max() < 0.2


def test_empty_and_unknown_observations():
    from fiducials_b200.node import FiducialSlam

    slam = FiducialSlam(max_fiducials=8)
    ident = [0, 0, 0, 0, 0, 0, 1]
    r = slam.transformCallback([], ident, ident)
    assert r.valid == 0 and slam.entries() == []
    slam.loadMap([[5, 0, 0, 0, 0, 0, 0, 0, 0]])
    obs = [dict(fiducial_id=9, translation=[0, 0, 1], rotation=[0, 0, 0, 1], image_error=0.1, object_error=1e-3, fiducial_area=100.0)]
    r = slam.transformCallback(obs, ident, ident)  # no known fiducial in view -> no pose, no map change
    assert r.valid == 0 and [e.fiducial_id for e in slam.entries()] == [5]
    r = slam.transformCallback(obs, None, None)  # tf lookup failed (map.cpp:270-273)
    assert r.valid == 0
    slam.clear()
    assert slam.entries() == []


def test_merge_matches_oracle_merge():
    from fiducials_b200 import _lib
    from fiducials_b200.node import FiducialSlam

    rng = np.random.default_rng(1)
    msgs, grid = _random_walk_messages(rng, 12, 60, 5)
    ident = so.TWV.identity()
    halves = [msgs[:30], msgs[30:]]
    slam = FiducialSlam(max_fiducials=32, n_instances=2)
    refs = []
    for inst, part in enumerate(halves):
        slam.loadMap([[100, grid[0][0], grid[0][1], grid[0][2], 180, 0, 180, 0, 0]], instance=inst)
        r = so.Map()
        r.load_entry(100, grid[0][0], grid[0][1], grid[0][2], 180, 0, 180, 0, 0)
        for m in part:
            r.update(so.observations_from_transforms(m), ident, ident)
        refs.append(r)
    slam.replay(halves, _tf7(ident), _tf7(ident))
    tables = np.concatenate([slam.export_table(0), slam.export_table(1)])
    local_before = [(e.fiducial_id, e.x, e.rz, e.variance, e.num_obs) for e in slam.entries(0)]
    slam.merge_tables(tables, 2)
    merged = so.merge_maps([[(f.id, f.pose, f.numObs) for f in r.fiducials.values()] for r in refs])

    def check(ents):
        assert [e.fiducial_id for e in ents] == sorted(merged)
        for e in ents:
            pose, n = merged[e.fiducial_id]
            rr = so.get_rpy(pose.R)
            assert np.abs(np.array([e.x, e.y, e.z]) - np.array(pose.t)).max() < 1e-9
            assert np.abs(np.array([e.rx, e.ry, e.rz]) - np.array(rr)).max() < 1e-9
            assert e.num_obs == n
            assert abs(e.variance - pose.var) <= 1e-9 * max(1.0, abs(pose.var))

    check(slam.merged_entries())
    # the merge writes a separate view: the local instances are untouched, so a second merge of the same
    # (re-exported) tables gives the same view (idempotence; round 1 folded the view back into the local map)
    assert [(e.fiducial_id, e.x, e.rz, e.variance, e.num_obs) for e in slam.entries(0)] == local_before
    first = [(e.fiducial_id, e.x, e.y, e.z, e.rx, e.ry, e.rz, e.variance, e.num_obs) for e in slam.merged_entries()]
    tables2 = np.concatenate([slam.export_table(0), slam.export_table(1)])
    assert np.array_equal(tables, tables2)
    slam.merge_tables(tables2, 2)
    assert [(e.fiducial_id, e.x, e.y, e.z, e.rx, e.ry, e.rz, e.variance, e.num_obs) for e in slam.merged_entries()] == first
    # explicit adoption: the view replaces an instance
    slam.adopt_merged(1)
    check(slam.entries(1))


def test_c5_pose_graph_sequence():
    """BASELINE.json config C5 (500 fiducials, ~10 observations per frame): the device fold equals the
    numpy restatement of Map::update over a 250-frame prefix, and the full 1000-frame sequence runs
    in one launch for several map instances at once."""
    from fiducials_b200 import synth
    from fiducials_b200.node import FiducialSlam

    msgs, seed_entry = synth.make_c5_sequence(1000, seed=0)
    ident = so.TWV.identity()
    ref = so.Map()
    ref.load_entry(*seed_entry)
    for m in msgs[:250]:
        ref.update(so.observations_from_transforms(m), ident, ident)
    slam = FiducialSlam(max_fiducials=512, n_instances=1)
    slam.loadMap([seed_entry])
    slam.replay([msgs[:250]], _tf7(ident), _tf7(ident))
    _cmp_entries(slam.entries(0), ref.entries(), 1e-4)  # BASELINE tolerance: 1e-4 m / 1e-4 rad
    _cmp_entries(slam.entries(0), ref.entries(), 1e-8)
    many = FiducialSlam(max_fiducials=512, n_instances=4)
    for i in range(4):
        many.loadMap([seed_entry], instance=i)
    many.replay([msgs] * 4, _tf7(ident), _tf7(ident))
    e0 = many.entries(0)
    assert len(e0) > 300  # the lawn-mower path has seen most of the ceiling
    for i in range(1, 4):
        ei = many.entries(i)
        assert [a.fiducial_id for a in ei] == [a.fiducial_id for a in e0]
        assert all(a.x == b.x and a.rz == b.rz for a, b in zip(ei, e0))  # deterministic across instances


def test_links_follow_the_fiducials(kat, tmp_path):
    """ADVICE r1: fiducials.clear() (clearCallback, map.cpp:809-817) drops the link sets with the fiducials; loadMap builds a
    fresh Fiducial for an id it replaces (map.cpp:600-606) -- no stale links may survive either on the device's slot x slot matrix."""
    from fiducials_b200.node import FiducialSlam

    tr = _bag_transforms(kat)
    ident = so.TWV.identity()
    slam = FiducialSlam(max_fiducials=32)
    slam.loadMap([[111, 0, 0, 0, 0, 0, 0, 0, 0]])
    for _ in range(3):
        slam.transformCallback(tr, _tf7(ident), _tf7(ident))
    links = slam.links()
    assert links and all(v for v in links.values())
    some = next(k for k in links if k != 111)
    # replacing one fiducial through loadMap: its own links and the links to it are gone, the others stay
    slam.loadMap([[some, 1, 2, 3, 0, 0, 0, 0.5, 0]])
    after = slam.links()
    assert some not in after and all(some not in v for v in after.values())
    assert any(after.values())
    # clear, then a different map: nothing of the old link matrix may show up under the new slot order
    slam.clear()
    assert slam.entries() == [] and slam.links() == {}
    slam.loadMap([[7, 0, 0, 0, 0, 0, 0, 0, 0], [9, 1, 0, 0, 0, 0, 0, 1, 0]])
    assert slam.links() == {}
    slam.close()


def test_load_map_file_with_tabs(tmp_path):
    """Map::loadMap's sscanf accepts tabs between the nine numbers; only the link list ends at the first tab (map.cpp:590-615)."""
    from fiducials_b200.node import FiducialSlam

    path = tmp_path / "tabs.txt"
    path.write_text("5\t1.0\t2.0 3.0\t0 0 90\t0.25\t4 6 7\textra words\n6 0 0 0 0 0 0 1 0 5\nnot a line\n7\t0\t0\t0\t0\t0\t0\t1\t2\n")
    slam = FiducialSlam(max_fiducials=8)
    assert slam.loadMapFile(str(path)) == 3
    ents = slam.entries()
    assert [e.fiducial_id for e in ents] == [5, 6, 7] and ents[0].num_obs == 4 and abs(ents[0].y - 2.0) < 1e-12 and abs(ents[0].rz - np.pi / 2) < 1e-12
    assert slam.links() == {5: [6, 7], 6: [5]}
    slam.close()


def test_messages_with_more_than_64_observations():
    """A FiducialTransformArray has no size limit (Map::update takes a std::vector<Observation>, map.cpp:152); round 1 clamped
    a message to 64 observations silently.  100 fiducials in every message, through all three entry points."""
    from fiducials_b200 import _lib
    from fiducials_b200.node import FiducialSlam

    rng = np.random.default_rng(5)
    n_fid = 100
    grid = [(float(i % 10), float(i // 10), 2.5) for i in range(n_fid)]
    msgs = []
    for k in range(6):
        cam = np.array([4.0 + 0.3 * k, 4.5 - 0.2 * k, 0.0])
        order = list(range(n_fid))
        rng.shuffle(order)
        m = []
        for i in order:
            t = np.array(grid[i]) - cam + rng.normal(0, 0.004, 3)
            q = so.q_from_rpy(math.pi + rng.normal(0, 0.01), rng.normal(0, 0.01), math.pi + rng.normal(0, 0.01))
            m.append(dict(fiducial_id=100 + i, translation=t, rotation=np.array(q), image_error=0.1, object_error=float(rng.uniform(1e-4, 1e-2)), fiducial_area=900.0))
        msgs.append(m)
    ident = so.TWV.identity()
    ref = so.Map()
    ref.load_entry(100, grid[0][0], grid[0][1], grid[0][2], 180, 0, 180, 0, 0)
    for m in msgs:
        ref.update(so.observations_from_transforms(m), ident, ident)
    assert len(ref.fiducials) == n_fid
    seed = [[100, grid[0][0], grid[0][1], grid[0][2], 180, 0, 180, 0, 0]]
    a = FiducialSlam(max_fiducials=128)
    a.loadMap(seed)
    for m in msgs:
        r = a.transformCallback(m, _tf7(ident), _tf7(ident))  # fid_map_update
    assert r.valid == 1 and r.n_estimates == n_fid
    _cmp_entries(a.entries(), ref.entries(), 1e-9)
    b = FiducialSlam(max_fiducials=128)
    b.loadMap(seed)
    b.replay([msgs], _tf7(ident), _tf7(ident))  # fid_map_update_sequence
    _cmp_entries(b.entries(), ref.entries(), 1e-9)
    assert b.links() == a.links() and len(a.links()[100]) == n_fid - 1
    # fid_map_update_frames: the dense per-frame layout of the detector (FID_MAX_MARKERS slots per frame)
    c = FiducialSlam(max_fiducials=128)
    c.loadMap(seed)
    from fiducials_b200.node import MAXM

    tfs = (_lib.fid_transform * (len(msgs) * MAXM))()
    counts = np.zeros(len(msgs), np.int32)
    for f, m in enumerate(msgs):
        counts[f] = len(m)
        arr = FiducialSlam._obs(m)
        for i in range(len(m)):
            tfs[f * MAXM + i] = arr[i]
    c.update_frames(counts, tfs, _tf7(ident), _tf7(ident))
    _cmp_entries(c.entries(), ref.entries(), 1e-9)
    for s in (a, b, c):
        s.close()


def test_add_fiducial_service():
    """add_fiducial (addFiducialCallback map.cpp:821-828, handleAddFiducial :489-535, called from every Map::update :173) on a
    read-only map: the requested id is inserted from the next message that observes it as T_mapBase * T_baseCam * T_camFid with
    the observation's variance; a request for an id that is already mapped is dropped; nothing else is added."""
    from fiducials_b200.node import FiducialSlam

    rng = np.random.default_rng(9)
    msgs, grid = _random_walk_messages(rng, 12, 20, 5)
    base_cam = so.TWV.from_qt(so.q_from_rpy(0.02, -0.03, 0.4), [0.1, -0.05, 0.3])
    cam_base = base_cam.inverse()
    map_base = so.TWV.from_qt(so.q_from_rpy(0.0, 0.0, 0.7), [1.5, -2.0, 0.0])
    seed = [100, grid[0][0], grid[0][1], grid[0][2], 180, 0, 180, 0, 0]
    ref = so.Map(read_only=True)
    ref.load_entry(*seed)
    slam = FiducialSlam(max_fiducials=32, read_only_map=True)
    slam.loadMap([seed])
    seen = sorted({t["fiducial_id"] for m in msgs for t in m} - {100})
    want, again = seen[0], seen[1]

    def step(m):
        r = ref.update(so.observations_from_transforms(m), base_cam, cam_base)
        g = slam.transformCallback(m, _tf7(base_cam), _tf7(cam_base))
        return r, g

    step(msgs[0])
    ref.fiducialToAdd, ref.addMapBase = want, map_base
    slam.addFiducial(want, _tf7(map_base))
    for m in msgs[1:8]:
        step(m)
    ref.fiducialToAdd, ref.addMapBase = again, None  # tf lookup failed: "Placing robot at the origin"
    slam.addFiducial(again, None)
    for m in msgs[8:14]:
        step(m)
    ref.fiducialToAdd, ref.addMapBase = want, None   # already in the map: the request is dropped
    slam.addFiducial(want, None)
    for m in msgs[14:]:
        step(m)
    assert ref.fiducialToAdd == -1
    ids = [e.fiducial_id for e in slam.entries()]
    assert ids == sorted(ref.fiducials) and set(ids) <= {100, want, again} and want in ids
    _cmp_entries(slam.entries(), ref.entries(), 1e-9)
    for e in slam.entries():
        assert abs(e.variance - ref.fiducials[e.fiducial_id].pose.var) <= 1e-9 * max(1.0, abs(e.variance))
    slam.close()


def test_batch_gauss_newton_refine_matches_oracle():
    """fid_map_refine (NEW, SURVEY 8f-3; parity unpinned -- the reference has no batch solver): the matrix-free PCG Gauss-Newton on the
    device lands on the poses of the dense numpy statement of the same problem (oracle/refine_oracle.py) -- same edges, weights,
    residuals, local parametrisation, damping and iteration count -- and the cost goes down monotonically from the sequential fold's map."""
    from fiducials_b200 import synth
    from fiducials_b200.node import FiducialSlam
    from oracle import refine_oracle as ro

    msgs, seed = synth.make_c5_sequence(120, seed=1, cols=6, rows=5, visible=6)
    ident = so.TWV.identity()
    slam = FiducialSlam(max_fiducials=64)
    slam.loadMap([seed])
    slam.replay([msgs], _tf7(ident), _tf7(ident))
    before = slam.entries()
    ids = [e.fiducial_id for e in before]
    R0 = [np.array(so.set_rpy_matrix(e.rx, e.ry, e.rz)) for e in before]
    t0 = [np.array([e.x, e.y, e.z]) for e in before]
    fixed = [e.variance == 0.0 for e in before]
    assert sum(fixed) == 1 and len(ids) == 30
    edges = ro.build_edges(ids, msgs)
    iters = 5
    Rr, tr, costs = ro.refine(R0, t0, fixed, edges, iterations=iters, damping=1e-6, lambda_t=2.0)
    st = slam.refine(msgs, max_iterations=iters, pcg_iterations=400, pcg_tolerance=1e-14, damping=1e-6, translation_weight=2.0)
    assert st.n_edges == len(edges) and st.n_free == 29 and st.iterations == iters
    assert abs(st.initial_cost - costs[0]) <= 1e-9 * costs[0] and abs(st.final_cost - costs[-1]) <= 1e-7 * costs[-1]
    assert st.final_cost < st.initial_cost and all(b <= a * (1 + 1e-12) for a, b in zip(costs, costs[1:]))
    after = slam.entries()
    assert [e.fiducial_id for e in after] == ids
    for e, R, t, f, b in zip(after, Rr, tr, fixed, before):
        assert np.abs(np.array([e.x, e.y, e.z]) - t).max() < 1e-7
        assert np.abs(np.array(so.set_rpy_matrix(e.rx, e.ry, e.rz)) - R).max() < 1e-7
        assert e.variance == b.variance and e.num_obs == b.num_obs  # only the poses move
        if f:
            assert (e.x, e.y, e.z, e.rx, e.ry, e.rz) == (b.x, b.y, b.z, b.rx, b.ry, b.rz)  # pinned entries stay put
    # the reference's map-quality metric (fiducial_slam/scripts/fit_plane.py) stays at the noise level of the observations
    assert ro.plane_fit_residual([[e.x, e.y, e.z] for e in after]) < 0.05
    slam.close()


def test_device_map_matches_the_reference_compiled_code():
    """The CUDA map update against the REFERENCE'S OWN Map class (fiducial_slam/src/map.cpp + transform_with_variance.cpp compiled
    unmodified against stand-in ROS / tf2 headers, oracle/Makefile) -- no restatement in between: per-message robot pose, the full
    C5 map and its links.  The reference's answers for this sequence are stored in tests/golden/map_ref_golden.npz
    (tests/golden/make_map_ref_golden.py)."""
    from fiducials_b200 import synth
    from fiducials_b200.node import FiducialSlam

    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "map_ref_golden.npz"))
    msgs, seed_entry = synth.make_c5_sequence(1000, seed=0)
    T_bc = [0.1, -0.02, 0.3, *so.q_from_rpy(0.02, -0.6, 0.1)]
    inv = so.TWV.from_qt(T_bc[3:], T_bc[:3]).inverse()
    T_cb = [*inv.t, *so.m_to_q(inv.R)]
    # message by message, with a camera offset: robot pose and variance of every update
    updates = gold["c5_updates"]  # rows: published, t[3], q[4], covariance diagonal[6]
    assert len(updates) == 120
    slam = FiducialSlam(max_fiducials=512)
    slam.loadMap([seed_entry])
    for m, u in zip(msgs[:120], updates):
        pub, t, q, cov = bool(u[0]), u[1:4], u[4:8], u[8:14]
        r = slam.transformCallback(m, np.array(T_bc), np.array(T_cb))
        assert bool(r.valid) == pub
        if pub:
            assert np.abs(np.array(r.t) - t).max() < 1e-9
            rq = np.array(r.q)
            assert min(np.abs(rq - q).max(), np.abs(rq + q).max()) < 1e-9
            assert abs(r.variance - cov[0]) <= 1e-9 * max(1.0, cov[0])
    re = gold["c5_k119_entries"]
    _cmp_entries(slam.entries(), [(int(x[0]), *x[1:7]) for x in re], 1e-9)
    ref_links = {}
    for a, b in gold["c5_k119_links"]:
        ref_links.setdefault(int(a), set()).add(int(b))
    assert {k: set(v) for k, v in slam.links().items()} == ref_links
    # the whole sequence in one launch against one replay inside the compiled reference
    one = FiducialSlam(max_fiducials=512)
    one.loadMap([seed_entry])
    ident = so.TWV.identity()
    one.replay([msgs], _tf7(ident), _tf7(ident))
    re = gold["c5_replay_entries"]
    assert len(re) == 500
    _cmp_entries(one.entries(0), [(int(x[0]), *x[1:7]) for x in re], 1e-8)
