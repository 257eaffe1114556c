"""Collision predicate on the CPU: the scene flattener, the oracle (alternating projections) against engine-independent
exact answers, and the product's GJK (csrc/gik_collide.cuh compiled for the host) against the oracle."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, rot_rpy

BOX, SPH, CYL = 0, 1, 2


def test_scene_matches_reference_construction(scene):
    # 45 robot primitives + table + obstacle + cube; 745 pairs = all cross-joint pairs - SRDF-disabled + (46, 47)
    assert len(scene.geoms) == 48 and len(scene.pairs) == 745
    assert (scene.table, scene.obstacle, scene.cube) == (45, 46, 47)
    assert [scene.geoms[i].name for i in (45, 46, 47)] == ["baseLink_0", "obstaclebase_0", "cubebase_0"]   # tools.py:40-41
    assert tuple(scene.pairs[-1]) == (46, 47)                                   # setup_pinocchio.py:58
    assert len(scene.obstacle_pairs()) == 78
    types = [g.type for g in scene.geoms[:45]]
    assert (types.count(BOX), types.count(CYL), types.count(SPH)) == (22, 19, 4)
    # translaterobot shifts only the first two geometries (setup_pinocchio.py:29-31)
    assert abs(scene.geoms[0].p[2] - (-0.435 + 0.85)) < 1e-12 and abs(scene.geoms[1].p[2] - (-0.82 + 0.85)) < 1e-12
    assert abs(scene.geoms[2].p[2] - (-0.82)) < 1e-12 and abs(scene.geoms[5].p[2] - 0.098) < 1e-12
    # no pair between geometries of the same joint; SRDF pairs absent
    for a, b in scene.pairs[:-1]:
        assert scene.geoms[a].joint != scene.geoms[b].joint
    links = {frozenset((scene.geoms[a].link, scene.geoms[b].link)) for a, b in scene.pairs}
    assert frozenset(("LARM_JOINT4_Link", "LARM_JOINT5_Link")) not in links
    assert frozenset(("CHEST_JOINT0_Link", "nextage_base")) not in links


def test_packaged_scene_equals_flattened_reference_urdfs(scene):
    # nextage_scene.json: reference_scene_from(<reference checkout>).to_json(), stored by tests/golden/make_golden.py
    ref = json.load(open(os.path.join(GOLDEN, "nextage_scene.json")))
    assert json.dumps(ref, sort_keys=True) == json.dumps(scene.to_json(), sort_keys=True)


def test_scene_from_urdf_geometry_order_placements_and_pairs(tmp_path):
    from gik_b200 import scene as sm
    from gik_b200.model import rpy_to_matrix

    def write(name, text):
        (tmp_path / name).write_text(text)
        return str(tmp_path / name)

    def col(shape, xyz="0 0 0"):
        return f'<collision><origin xyz="{xyz}"/><geometry>{shape}</geometry></collision>'

    box, sph, cyl = '<box size="0.2 0.4 0.6"/>', '<sphere radius="0.05"/>', '<cylinder radius="0.1" length="0.4"/>'
    # children are visited in joint-name order (J0 before J1); a fixed joint's geometry joins its parent joint
    robot = write("r.urdf", f"""<robot name="r">
      <link name="base">{col(box, "0 0 0.1")}{col(sph)}{col(cyl, "0 0 -0.3")}</link>
      <link name="l1">{col(cyl)}</link><link name="l1b">{col(box, "0.1 0 0")}</link><link name="l0">{col(sph, "0.1 0 0")}</link>
      <joint name="J1" type="revolute"><parent link="base"/><child link="l1"/><origin xyz="0 1 0"/><axis xyz="0 0 1"/></joint>
      <joint name="F" type="fixed"><parent link="l1"/><child link="l1b"/><origin xyz="0 0 0.5" rpy="0 0 1.5708"/></joint>
      <joint name="J0" type="revolute"><parent link="base"/><child link="l0"/><origin xyz="1 0 0"/><axis xyz="1 0 0"/></joint>
    </robot>""")
    srdf = write("r.srdf", '<robot name="r"><disable_collisions link1="l1b" link2="l0" reason="Adjacent"/></robot>')
    table = write("t.urdf", f'<robot name="t"><link name="baseLink">{col(box, "0 0 0.2")}</link></robot>')
    obstacle = write("o.urdf", f'<robot name="o"><link name="obstaclebase">{col(sph)}</link></robot>')
    cube = write("c.urdf", '<robot name="c"><link name="cubebase"><collision><geometry><mesh filename="cube.stl" '
                           'scale="0.04 0.04 0.04"/></geometry></collision></link></robot>')
    rz = rpy_to_matrix([0, 0, -np.pi / 2])
    s = sm.scene_from_urdf(robot, srdf, table, obstacle, cube, robot_placement=(np.eye(3), np.array([0, 0, 0.85])),
                           table_placement=(rz, np.array([0.8, 0, 0])), obstacle_placement=(np.eye(3), np.array([0.4, 0, 0.9])),
                           cube_placement=(np.eye(3), np.array([0.33, -0.3, 0.93])))
    assert [g.name for g in s.geoms] == ["base_0", "base_1", "base_2", "l0_0", "l1_0", "l1b_0", "baseLink_0",
                                         "obstaclebase_0", "cubebase_0"]
    assert [g.joint for g in s.geoms] == [-1, -1, -1, 0, 1, 1, -1, -1, -1]
    assert [g.type for g in s.geoms] == [BOX, SPH, CYL, SPH, CYL, BOX, BOX, SPH, BOX]
    assert (s.table, s.obstacle, s.cube) == (6, 7, 8)
    assert np.allclose(s.geoms[0].size, [0.1, 0.2, 0.3]) and np.allclose(s.geoms[1].size, [0.05, 0, 0])
    assert np.allclose(s.geoms[2].size, [0.1, 0.2, 0]) and np.allclose(s.geoms[8].size, [0.02, 0.02, 0.02])
    # the robot placement moves only the first two root geometries
    assert np.allclose(s.geoms[0].p, [0, 0, 0.95]) and np.allclose(s.geoms[1].p, [0, 0, 0.85])
    assert np.allclose(s.geoms[2].p, [0, 0, -0.3])
    # moving-joint geometries are expressed in their joint's frame, fixed-joint offsets composed in
    assert np.allclose(s.geoms[3].p, [0.1, 0, 0]) and np.allclose(s.geoms[4].p, 0)
    assert np.allclose(s.geoms[5].p, [0, 0.1, 0.5], atol=1e-5) and np.allclose(s.geoms[5].R, rpy_to_matrix([0, 0, 1.5708]))
    assert np.allclose(s.geoms[6].p, [0.8, 0, 0.2]) and np.allclose(s.geoms[6].R, rz)
    assert np.allclose(s.geoms[7].p, [0.4, 0, 0.9]) and np.allclose(s.geoms[8].p, [0.33, -0.3, 0.93])
    # all pairs on different joints, minus the SRDF-disabled (l0, l1b), plus (obstacle, cube)
    assert [tuple(p) for p in s.pairs] == [(0, 3), (0, 4), (0, 5), (1, 3), (1, 4), (1, 5), (2, 3), (2, 4), (2, 5), (3, 4),
                                           (3, 6), (3, 7), (3, 8), (4, 6), (4, 7), (4, 8), (5, 6), (5, 7), (5, 8), (7, 8)]
    assert json.dumps(sm.CollisionScene.from_json(s.to_json()).to_json()) == json.dumps(s.to_json())


def test_oracle_pair_distances_against_closed_forms(c_oracle):
    I = np.eye(3)
    # box-box, axis aligned: gap along x
    d = c_oracle.pair_distance(BOX, I, [0, 0, 0], [1, 1, 1], BOX, I, [3, 0.5, 0], [0.5, 0.5, 0.5])
    assert abs(d - 1.5) < 1e-9
    # sphere-sphere
    d = c_oracle.pair_distance(SPH, I, [0, 0, 0], [0.5, 0, 0], SPH, I, [0, 2, 0], [0.25, 0, 0])
    assert abs(d - 1.25) < 1e-9
    # sphere above a rotated box corner-on: distance to the face through closed form (face normal direction)
    R = rot_rpy(0, 0, 0.7)
    d = c_oracle.pair_distance(BOX, R, [0, 0, 0], [1, 2, 0.5], SPH, I, [0, 0, 2], [0.3, 0, 0])
    assert abs(d - (2 - 0.5 - 0.3)) < 1e-9
    # cylinder (axis z) next to a sphere: radial gap
    d = c_oracle.pair_distance(CYL, I, [0, 0, 0], [0.2, 1.0, 0], SPH, I, [1, 0, 0.3], [0.1, 0, 0])
    assert abs(d - (1 - 0.2 - 0.1)) < 1e-9
    # two parallel cylinders
    d = c_oracle.pair_distance(CYL, I, [0, 0, 0], [0.2, 1.0, 0], CYL, I, [0.7, 0, 0.5], [0.3, 1.0, 0])
    assert abs(d - 0.2) < 1e-9
    # crossed cylinders (axes z and x), centres 1 apart along y
    Rx = rot_rpy(0, np.pi / 2, 0)
    d = c_oracle.pair_distance(CYL, I, [0, 0, 0], [0.2, 1.0, 0], CYL, Rx, [0, 1, 0], [0.3, 1.0, 0])
    assert abs(d - 0.5) < 1e-9
    # overlapping -> 0
    assert c_oracle.pair_distance(BOX, R, [0, 0, 0], [1, 1, 1], CYL, Rx, [1.2, 0, 0], [0.3, 0.5, 0]) == 0.0


def _random_shape(rng, scale=1.0):
    t = int(rng.integers(0, 3))
    R = rot_rpy(*rng.uniform(-np.pi, np.pi, 3))
    size = np.zeros(3)
    if t == BOX:
        size[:] = rng.uniform(0.05, 0.4, 3)
    elif t == SPH:
        size[0] = rng.uniform(0.05, 0.3)
    else:
        size[:2] = rng.uniform(0.05, 0.3), rng.uniform(0.05, 0.4)
    return t, R, size * scale


@pytest.mark.parametrize("dtype,band", [(np.float64, 1e-6), (np.float32, 1e-4)])
def test_gjk_agrees_with_projection_oracle_on_random_pairs(hostsim, c_oracle, dtype, band):
    rng = np.random.default_rng(7)
    checked = hits = 0
    for _ in range(1500):
        ta, Ra, sa = _random_shape(rng)
        tb, Rb, sb = _random_shape(rng)
        pa = rng.uniform(-0.3, 0.3, 3)
        pb = pa + rng.normal(size=3) * rng.uniform(0.05, 0.7)
        d = c_oracle.pair_distance(ta, Ra, pa, sa, tb, Rb, pb, sb)
        got = hostsim.pair(ta, Ra, pa, sa, tb, Rb, pb, sb, dtype)
        if 0.0 < d < band:
            continue                       # grazing contact: either answer is within round-off of the truth
        if d == 0.0:
            # the oracle cannot tell touching from overlapping: confirm a real overlap by shrinking A a little
            d_shrunk = c_oracle.pair_distance(ta, Ra, pa, sa * 0.98, tb, Rb, pb, sb * 0.98)
            if d_shrunk > 0.0:
                continue
        checked += 1
        hits += int(d == 0.0)
        assert got == (d == 0.0), (ta, tb, d)
        # margin: "closer than m" <=> inflated intersection
        if d > band:
            assert hostsim.pair(ta, Ra, pa, sa, tb, Rb, pb, sb, dtype, margin=d * 1.05 + 10 * band)
            assert not hostsim.pair(ta, Ra, pa, sa, tb, Rb, pb, sb, dtype, margin=max(d * 0.95 - 10 * band, 0.0)) or d < 20 * band
    assert checked > 1200 and 200 < hits < 1300


def test_reference_known_answers(table_c, scene_c, c_oracle, hostsim, golden):
    # collision(robot, q0) == True (lab_instructions.ipynb:252)
    assert c_oracle.scene_distance(table_c, scene_c, np.zeros((1, 15)))[0] == 0.0
    assert hostsim.collide(table_c, scene_c, np.zeros((1, 15)), None, np.float64)[0]
    # the two recorded grasp poses were accepted by the reference (success=True): collision-free, hand boxes 1 mm off the cube
    Q = np.array([c["q"] for c in golden["cases"]])
    P = np.array([c["cube_R"] + c["cube_p"] for c in golden["cases"]], float)
    d = c_oracle.scene_distance(table_c, scene_c, Q, P)
    assert (d > 5e-4).all() and (d < 1.5e-3).all()
    for dt in (np.float64, np.float32):
        assert not hostsim.collide(table_c, scene_c, Q, P, dt).any()
    # cube resting 5 mm above the table top at both placements (config.py:36-37), not touching the obstacle
    dc = c_oracle.scene_distance(table_c, scene_c, None, P, mode=2)
    assert np.abs(dc - 0.005).max() < 1e-9
    assert not hostsim.collide(table_c, scene_c, None, P, np.float64, mode=2).any()


def test_full_scene_gjk_vs_oracle(table, table_c, scene_c, c_oracle, hostsim):
    rng = np.random.default_rng(11)
    n = 160
    Q = rng.uniform(table.lower, table.upper, size=(n, 15)) * 0.7
    P = np.zeros((n, 12)); P[:, [0, 4, 8]] = 1
    P[:, 9:] = rng.uniform([0.2, -0.4, 0.93], [0.6, 0.4, 1.4], size=(n, 3))
    d_all = c_oracle.scene_distance(table_c, scene_c, Q, P, mode=0, cull=0.05)
    d_obs = c_oracle.scene_distance(table_c, scene_c, Q, P, mode=1, cull=0.2)
    for dt, band in ((np.float64, 1e-6), (np.float32, 1e-4)):
        got = hostsim.collide(table_c, scene_c, Q, P, dt)
        sure = (d_all == 0) | (d_all > band)
        assert sure.mean() > 0.9 and (got[sure] == (d_all[sure] == 0)).all()
        near = hostsim.collide(table_c, scene_c, Q, P, dt, mode=1, margin=0.04)      # distanceToObstacle < 0.04
        sure = np.abs(d_obs - 0.04) > 10 * band
        assert (near[sure] == (d_obs[sure] < 0.04)).all()
    assert 0.05 < (d_all == 0).mean() < 0.98
    # cube-only test over placements around the obstacle and the table top
    Pc = np.zeros((200, 12)); Pc[:, [0, 4, 8]] = 1
    Pc[:, 9:] = rng.uniform([0.2, -0.3, 0.85], [0.65, 0.15, 1.1], size=(200, 3))
    Pc[::3, :9] = rot_rpy(0, 0, 0.6).reshape(9)
    dc = c_oracle.scene_distance(table_c, scene_c, None, Pc, mode=2)
    got = hostsim.collide(table_c, scene_c, None, Pc, np.float64, mode=2)
    sure = (dc == 0) | (dc > 1e-6)
    assert (got[sure] == (dc[sure] == 0)).all() and 0.1 < got.mean() < 0.9
