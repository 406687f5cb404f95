"""The reference's own problem files, loaded VERBATIM (tests/golden/reference_json/*.json are byte copies of
trajopt_common/data/config/{arm_around_table,simple_collision_test,numerical_ik1,box_cast_test}.json) through the JSON
front end and solved.  What the files do not carry — the tesseract environment — is replaced by this repo's fixtures:
the PR2 arm chains and spherebot of robots.py (constants of the reference's URDFs) and sphere worlds (the reference's
scenes are meshes / boxes through Bullet: SURVEY.md section 8f).  arm_around_table.json runs with its own
longest_valid_segment_length of 0.02: ~38 sub-segments per step pair (the sub-trajectory is unbounded, as in the reference).
CPU: the oracle solves them and meets the reference tests' expectations.  GPU: the CUDA path gives the oracle's answer."""
import hashlib
import os

import numpy as np
import pytest

from trajopt_b200 import capi, json_io, robots

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_json")
ARM_START = [-1.832, -0.332, -1.011, -1.437, -1.1, -1.926, 3.074]
TABLE = np.array([[[0.75, -0.2, 0.45, 0.10]]])  # one obstacle sphere under the arm's path (the file's margin buffer is the JSON
# default of 0.5 m: nearly all of the 7 x 38 candidates of a step pair are active contacts)


def _load(name):
    doc = open(os.path.join(G, name + ".json")).read()
    if name == "arm_around_table":
        return json_io.from_json(doc, robots.pr2_arm("r", with_spheres=True), np.array([ARM_START]), obstacles=TABLE)
    if name == "simple_collision_test":
        return json_io.from_json(doc, robots.spherebot(), np.array([[-0.75, 0.75]]), obstacles=robots.SPHEREBOT_OBSTACLES[None])
    if name == "numerical_ik1":
        return json_io.from_json(doc, robots.pr2_arm("l", with_spheres=False), np.zeros((1, 7)))
    if name == "box_cast_test":  # boxbot's two prismatic joints = spherebot's; one obstacle on the straight path
        return json_io.from_json(doc, robots.spherebot(), np.array([[-1.9, 0.0]]), obstacles=np.array([[[0.0, 1.0, 0.0, 0.4]]]))
    raise KeyError(name)


NAMES = ["arm_around_table", "simple_collision_test", "numerical_ik1", "box_cast_test"]


def test_files_are_the_reference_bytes():
    """tests/golden/reference_json.sha256 holds the SHA-256 of the reference's own files (trajopt v0.35.0,
    `sha256sum` run in trajopt_common/data/config): the copies here must hash to the same values."""
    want = dict(reversed(line.split()) for line in open(G + ".sha256").read().splitlines())
    assert sorted(want) == sorted(n + ".json" for n in NAMES)
    for n in NAMES:
        assert hashlib.sha256(open(os.path.join(G, n + ".json"), "rb").read()).hexdigest() == want[n + ".json"], n


def test_arm_around_table_keeps_its_lvs(oracle):
    d = _load("arm_around_table")
    coll = [t for t in d.terms if t.kind == capi.TERM_COLLISION][0]
    assert coll.longest_valid_segment_length == 0.02 and coll.evaluator_type == capi.COLL_LVS_CONTINUOUS
    assert list(coll.fixed_steps[:coll.n_fixed_steps]) == [0, 5]
    step = np.linalg.norm(np.diff(d.init_traj[0], axis=0), axis=1)
    assert np.ceil(step / 0.02).max() >= 30  # far beyond the cap of 4 sub-segments this path used to have
    r = oracle.solve_batch(d)
    assert r["status"][0] == capi.OPT_CONVERGED
    np.testing.assert_allclose(r["x"][0, 0], ARM_START, atol=1e-9)                                       # fixed_timesteps
    np.testing.assert_allclose(r["x"][0, 5], [0.062, 1.287, 0.1, -1.554, -3.011, -0.268, 2.988], atol=1e-3)  # joint_pos cnt


def test_simple_collision_leaves_collision(oracle):
    """simple_collision_unit.cpp:60-123: spherebot starts in collision and must end collision free."""
    d = _load("simple_collision_test")
    r = oracle.solve_batch(d)
    assert r["status"][0] == capi.OPT_CONVERGED
    q = r["x"][0, 0]
    c = np.array([q[0], q[1], 0.0])
    dist = np.linalg.norm(robots.SPHEREBOT_OBSTACLES[:, :3] - c, axis=1) - robots.SPHEREBOT_OBSTACLES[:, 3] - 0.5
    assert (dist > 0.2 - 1e-3).all(), dist  # outside the constraint's dist_pen


def test_numerical_ik_reaches_the_pose(oracle):
    """numerical_ik_unit.cpp:60-124: every entry of the final tool pose within 1e-3 of the goal."""
    d = _load("numerical_ik1")
    r = oracle.solve_batch(d)
    la = robots.pr2_arm("l", with_spheres=False)
    R, p = robots.fk_numpy(la, r["x"][0, 0])[la["tool"]]
    np.testing.assert_allclose(p, [0.4, 0.0, 0.8], atol=1e-3)
    np.testing.assert_allclose(R, np.diag([-1.0, 1.0, -1.0]), atol=1e-3)  # wxyz (0,0,1,0): half turn about y


def test_box_cast_clears_the_obstacle(oracle):
    """cast_cost_unit.cpp:60-117 shape: the straight path crosses the obstacle, the cast cost pushes it out."""
    d = _load("box_cast_test")
    r = oracle.solve_batch(d)
    x = r["x"][0]
    np.testing.assert_allclose(x[0], [-1.9, 0.0], atol=1e-9)
    np.testing.assert_allclose(x[2], [1.9, 3.8], atol=1e-3)
    ts = np.linspace(0, 1, 50)[:, None]
    for a, b in ((x[0], x[1]), (x[1], x[2])):  # swept centre against the obstacle
        c = np.c_[a + (b - a) * ts, np.zeros(50)]
        assert (np.linalg.norm(c - [0.0, 1.0, 0.0], axis=1) - 0.4 - 0.5 > -1e-3).all()


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_cuda_solves_the_reference_files(oracle, name):
    from trajopt_b200 import api
    d = _load(name)
    got = api.solve(d)
    ref = oracle.solve_batch(d)
    assert got["status"][0] == ref["status"][0] and got["n_qp_solves"][0] == ref["n_qp_solves"][0]
    np.testing.assert_allclose(got["total_cost"], ref["total_cost"], atol=1e-6)
    np.testing.assert_allclose(got["cnt_viols"], ref["cnt_viols"], atol=1e-6)
    # numerical_ik1 has no cost and 6 pose equations for 7 joints: every QP has a one-dimensional set of minimisers, and
    # where ADMM stops along it is decided at the 1e-10 level of its linear solves (the reference's own test,
    # numerical_ik_unit.cpp, checks the end pose only).  The other files have strictly convex QPs.
    np.testing.assert_allclose(got["x"], ref["x"], atol=1e-4 if name == "numerical_ik1" else 1e-5)
