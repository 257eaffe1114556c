"""Regenerates the committed fixtures from the reference checkout (run in the build container only):

    python tests/golden/make_golden.py [/root/reference]

  ik_golden.json      -- the reference's own recorded outputs of computeqgrasppose (config 1):
                         trajectory.json / trajectory2.json `q_control_points[0]` and `[-1]` are q0 and qe,
                         pinned there by the SLSQP equality constraints of control.py:110-119 and produced at
                         control.py:435-436; plus the notebook known answers (lab_instructions.ipynb:210-226,
                         252, 290-293) typed from the recorded cell outputs.
  trajectory2_reference.json -- trajectory2.json as saved by control.save_trajectory_to_json (control.py:203-216):
                         the control points of a maketraj result and of its two derivative curves.
  nextage_table.json  -- the kinematic table flattened from the reference's URDFs
                         (models/nextagea_description/urdf/NextageaOpen.urdf, models/cubes/cube_small.urdf)
                         with ROBOT_PLACEMENT (config.py:33) applied as in setup_pinocchio.py:28-32.
  nextage_scene.json  -- the collision scene flattened from the reference's URDF/SRDF files (scene.reference_scene_from);
                         the package ships the same file as data/nextage_scene.json.
The fixtures are data; no reference source code is copied."""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))


def main(ref):
    t1 = json.load(open(os.path.join(ref, "trajectory.json")))
    t2 = json.load(open(os.path.join(ref, "trajectory2.json")))
    assert t1["q_control_points"][0] == t2["q_control_points"][0]
    assert t1["q_control_points"][-1] == t2["q_control_points"][-1]
    gold = {
        "source": "trajectory.json / trajectory2.json q_control_points[0], [-1]; lab_instructions.ipynb outputs",
        "q_init": [0.0] * 15,
        "cases": [
            {"name": "q0", "cube_R": [1, 0, 0, 0, 1, 0, 0, 0, 1], "cube_p": [0.33, -0.3, 0.93],   # config.py:36
             "q": t1["q_control_points"][0], "success": True, "iterations_chart": 740},
            {"name": "qe", "cube_R": [1, 0, 0, 0, 1, 0, 0, 0, 1], "cube_p": [0.4, 0.11, 0.93],    # config.py:37
             "q": t1["q_control_points"][-1], "success": True, "iterations_chart": 736},
        ],
        "notebook": {
            "joint_names": ["universe", "CHEST_JOINT0", "HEAD_JOINT0", "HEAD_JOINT1", "LARM_JOINT0", "LARM_JOINT1",
                            "LARM_JOINT2", "LARM_JOINT3", "LARM_JOINT4", "LARM_JOINT5", "RARM_JOINT0", "RARM_JOINT1",
                            "RARM_JOINT2", "RARM_JOINT3", "RARM_JOINT4", "RARM_JOINT5"],
            "oMf_LARM_EFF_at_q0": {"R": [[-3.67321e-06, -1, 0], [1, -3.67321e-06, 0], [0, 0, 1]],
                                   "p": [0.452, 0.28, 0.851], "print_precision": 6},
            "collision_at_q0": True,
        },
    }
    json.dump(gold, open(os.path.join(HERE, "ik_golden.json"), "w"), indent=1)
    json.dump(t2, open(os.path.join(HERE, "trajectory2_reference.json"), "w"))     # the reference's saved maketraj result
    import gik_b200
    tab = gik_b200.from_urdf(os.path.join(ref, "models/nextagea_description/urdf/NextageaOpen.urdf"),
                             os.path.join(ref, "models/cubes/cube_small.urdf"))
    json.dump(tab.to_json(), open(os.path.join(HERE, "nextage_table.json"), "w"), indent=1)
    from gik_b200 import scene
    sc = scene.reference_scene_from(ref).to_json()
    json.dump(sc, open(os.path.join(HERE, "nextage_scene.json"), "w"))
    os.makedirs(os.path.join(HERE, "..", "..", "motion-planning-and-control-for-dual-manipulator-robot_b200", "data"), exist_ok=True)
    json.dump(sc, open(os.path.join(HERE, "..", "..", "motion-planning-and-control-for-dual-manipulator-robot_b200", "data",
                                    "nextage_scene.json"), "w"))
    print("wrote ik_golden.json, trajectory2_reference.json, nextage_table.json, nextage_scene.json, data/nextage_scene.json")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "/root/reference")
