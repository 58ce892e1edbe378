"""MJCF scene composer + compiler for the furniture-assembly scene family.

Two jobs, both host-side Python (the reference's composer is Python too):

1. ``compose_scene`` restates the reference's scene composition: base world + floor arena +
   robot (+ gripper mounted under ``right_hand``) + furniture parts (free joint, friction,
   origin site) + weld equalities, producing one MJCF string -- the same string the reference
   hands to ``load_model_from_xml``.
     reference: furniture/env/models/base.py:76-101 (merge), models/robots/robot.py:15-46
     (add_gripper), models/tasks/floor_task.py:18-72 (merge order, free joint damping 0.0001),
     models/objects/objects.py:186-206 (get_collision: friction 1 10 0.5, origin site),
     models/arenas/arena.py:86-103 (floor size/friction), furniture.py:1889-2031 (_load_model_*).

2. ``compile_mjcf`` is a small MJCF compiler for the feature subset those scenes use (SURVEY.md
   A.3): fixed/hinge/slide/free joints, explicit <inertial> or density-derived inertia of
   box/cylinder/sphere/capsule geoms, plane/box/cylinder/sphere/capsule colliders, sites,
   motor/position/velocity actuators, weld equalities, <default> classes, <contact><exclude>.
   It replaces ``mujoco_py.load_model_from_xml`` (models/base.py:113-115) and returns a flat
   table ``Model`` that both the CPU oracle and the CUDA engine ingest.

Nothing here is on the per-step hot path.
"""
from __future__ import annotations

import copy
import glob
import io
import math
import os
import xml.etree.ElementTree as ET
from dataclasses import dataclass, field

import numpy as np

# --------------------------------------------------------------------------------------
# small quaternion helpers (w, x, y, z)
# --------------------------------------------------------------------------------------


def q_mul(a, b):
    aw, ax, ay, az = a
    bw, bx, by, bz = b
    return np.array(
        [
            aw * bw - ax * bx - ay * by - az * bz,
            aw * bx + ax * bw + ay * bz - az * by,
            aw * by - ax * bz + ay * bw + az * bx,
            aw * bz + ax * by - ay * bx + az * bw,
        ]
    )


def q_conj(q):
    return np.array([q[0], -q[1], -q[2], -q[3]])


def q_norm(q):
    q = np.asarray(q, dtype=np.float64)
    n = np.linalg.norm(q)
    if n < 1e-14:
        return np.array([1.0, 0.0, 0.0, 0.0])
    return q / n


def q_to_mat(q):
    w, x, y, z = q
    return np.array(
        [
            [w * w + x * x - y * y - z * z, 2 * (x * y - w * z), 2 * (x * z + w * y)],
            [2 * (x * y + w * z), w * w - x * x + y * y - z * z, 2 * (y * z - w * x)],
            [2 * (x * z - w * y), 2 * (y * z + w * x), w * w - x * x - y * y + z * z],
        ]
    )


def q_axis_angle(axis, angle):
    axis = np.asarray(axis, dtype=np.float64)
    s = math.sin(angle * 0.5)
    return np.array([math.cos(angle * 0.5), axis[0] * s, axis[1] * s, axis[2] * s])


def mat_to_q(R):
    """Rotation matrix -> unit quaternion (w,x,y,z)."""
    t = np.trace(R)
    if t > 0:
        s = math.sqrt(t + 1.0) * 2
        q = np.array([0.25 * s, (R[2, 1] - R[1, 2]) / s, (R[0, 2] - R[2, 0]) / s, (R[1, 0] - R[0, 1]) / s])
    elif R[0, 0] > R[1, 1] and R[0, 0] > R[2, 2]:
        s = math.sqrt(1.0 + R[0, 0] - R[1, 1] - R[2, 2]) * 2
        q = np.array([(R[2, 1] - R[1, 2]) / s, 0.25 * s, (R[0, 1] + R[1, 0]) / s, (R[0, 2] + R[2, 0]) / s])
    elif R[1, 1] > R[2, 2]:
        s = math.sqrt(1.0 + R[1, 1] - R[0, 0] - R[2, 2]) * 2
        q = np.array([(R[0, 2] - R[2, 0]) / s, (R[0, 1] + R[1, 0]) / s, 0.25 * s, (R[1, 2] + R[2, 1]) / s])
    else:
        s = math.sqrt(1.0 + R[2, 2] - R[0, 0] - R[1, 1]) * 2
        q = np.array([(R[1, 0] - R[0, 1]) / s, (R[0, 2] + R[2, 0]) / s, (R[1, 2] + R[2, 1]) / s, 0.25 * s])
    return q_norm(q)


def euler_xyz_to_q(e):
    """MJCF default eulerseq "xyz": intrinsic rotations about x, then y', then z''."""
    qx = q_axis_angle([1, 0, 0], e[0])
    qy = q_axis_angle([0, 1, 0], e[1])
    qz = q_axis_angle([0, 0, 1], e[2])
    return q_mul(q_mul(qx, qy), qz)


# --------------------------------------------------------------------------------------
# constants shared with the C oracle and the CUDA engine
# --------------------------------------------------------------------------------------
JNT_FREE, JNT_SLIDE, JNT_HINGE = 0, 2, 3  # numeric values follow mjtJoint (ball=1 unused)
GEOM_PLANE, GEOM_SPHERE, GEOM_CAPSULE, GEOM_CYLINDER, GEOM_BOX, GEOM_MESH = 0, 2, 3, 5, 6, 7  # mjtGeom
GEOM_TYPES = {"plane": GEOM_PLANE, "sphere": GEOM_SPHERE, "capsule": GEOM_CAPSULE, "cylinder": GEOM_CYLINDER, "box": GEOM_BOX}
ACT_MOTOR, ACT_POSITION, ACT_VELOCITY = 0, 1, 2

MJ_MINVAL = 1e-15


def _floats(s, n=None, default=None):
    if s is None:
        return None if default is None else np.array(default, dtype=np.float64)
    v = np.array([float(x) for x in s.split()], dtype=np.float64)
    if n is not None and v.size < n and default is not None:
        d = np.array(default, dtype=np.float64)
        d[: v.size] = v
        v = d
    return v


# --------------------------------------------------------------------------------------
# scene composition (reference composer restated)
# --------------------------------------------------------------------------------------

def default_assets_root():
    """the reference's MJCF asset tree (furniture/env/models/assets) named by FURNITURE_ASSETS, or None"""
    cand = os.environ.get("FURNITURE_ASSETS")
    return cand if cand and os.path.isdir(cand) else None


def furniture_names(assets_root):
    """Sorted furniture names; the index is the reference's furniture_id (models/__init__.py:10-22)."""
    xmls = sorted(glob.glob(os.path.join(assets_root, "objects", "*.xml")))
    return [os.path.basename(x).split(".")[0] for x in xmls]


def _section(root, name):
    found = root.find(name)
    if found is None:
        found = ET.SubElement(root, name)
    return found


def _merge(dst_root, src_root, merge_body=True):
    """MujocoXML.merge (models/base.py:76-101): worldbody children, asset (dedup by tag+name),
    actuator, equality, sensor, contact, default -- nothing else (<option>, <compiler>, <size> of the
    merged file are dropped, SURVEY.md A.2)."""
    if merge_body:
        for child in list(_section(src_root, "worldbody")):
            _section(dst_root, "worldbody").append(child)
    dst_asset = _section(dst_root, "asset")
    for a in list(_section(src_root, "asset")):
        nm = a.get("name")
        if nm is None or dst_asset.find("./{}[@name='{}']".format(a.tag, nm)) is None:
            dst_asset.append(a)
    for sec in ("actuator", "equality", "sensor", "contact", "default"):
        for child in list(_section(src_root, sec)):
            _section(dst_root, sec).append(child)


SAWYER_INIT_QPOS = np.array([-0.28, -0.60, 0.00, 1.86, 0.00, 0.3, 1.57])  # robots/sawyer_robot.py:20
SAWYER_BOTTOM_OFFSET = np.array([0.0, 0.0, -0.913])  # robots/sawyer_robot.py:17
BAXTER_INIT_QPOS = np.array([0.814, -0.44, -0.07, 0.5, 0, 1.641, -1.57629266, -0.872, -0.39, 0.07, 0.5, 0, 1.641, -1.57629197])  # robots/baxter_robot.py:45-47
BAXTER_BOTTOM_OFFSET = np.array([0.0, 0.0, -0.913])  # robots/baxter_robot.py:19
GRIPPER_INIT_QPOS = np.array([0.020833, -0.020833])  # grippers/two_finger_gripper.py:22-23


def place_unlisted_parts(part_names, listed, radii, seed):
    """Base placement of the parts whose XML carries no `<name>_initpos` numeric (7 of the shipped furniture models).
    Restates UniformRandomSampler.setup (models/tasks/placement_sampler.py:68-104 with the (0.7, 0.7, 0) table of
    floor_task.py:37): such a part starts from Qpos(0, 0, 0, identity) and is drawn once, at construction, uniformly in
    +-0.35 m in x and y, 0.01 above, rejecting draws whose horizontal-radius disc overlaps a part already placed
    (the XML-listed parts count as placed).  Every reset then jitters around that base like any listed part.
    The reference draws from the env's numpy RandomState at construction; here the draw is part of scene composition
    (one RandomState(seed) per composed scene) so that engine, oracle and tests see the same base poses."""
    rng = np.random.RandomState(int(seed) & 0x7FFFFFFF)
    placed = [(q[0], q[1], radii.get(n, 0.0)) for n, q in listed.items()]
    out = {}
    for name in part_names:
        if name in listed:
            continue
        r = radii.get(name, 0.0)
        for _ in range(10000):
            x, y = rng.uniform(-0.35, 0.35), rng.uniform(-0.35, 0.35)
            if all(np.hypot(x - px, y - py) > pr + r for px, py, pr in placed):
                break
        else:
            raise RuntimeError("cannot place all parts on the floor")  # RandomizationError, placement_sampler.py:187
        placed.append((x, y, r))
        out[name] = np.array([x, y, 0.01, 1.0, 0.0, 0.0, 0.0])
    return out


def _rescale_objects(obj_root, mult):
    """xml_adjusting/rescale.py:30-95 (`rescale`, used by MujocoXMLObject(resize=...), objects.py:136-147): mesh scales of the part
    meshes, body positions, and every site / geom position and size under the part bodies are multiplied by `mult`; the
    `*_initpos` numerics and the weld data are left alone, as in the reference."""
    def mul(sv):
        return " ".join(str(float(x) * mult) for x in sv.split())

    asset = obj_root.find("asset")
    if asset is not None:
        for mesh in asset:
            if mesh.tag == "mesh" and "part" in mesh.get("name", ""):
                mesh.set("scale", mul(mesh.get("scale", "1 1 1")))
    for body in obj_root.find("worldbody"):
        if "_part" in body.get("name", ""):
            body.set("pos", mul(body.get("pos", "0 0 0")))
            for child in body.iter():
                if child.tag == "site":
                    child.set("pos", mul(child.get("pos", "0 0 0")))
                    if child.get("size") is not None:
                        child.set("size", mul(child.get("size")))
                elif child.tag == "geom":
                    if child.get("pos") is not None:
                        child.set("pos", mul(child.get("pos")))
                    if child.get("size") is not None:
                        child.set("size", mul(child.get("size")))


def compose_scene(agent="Sawyer", furniture="table_lack_0825", assets_root=None, use_torque=False, placement_seed=123, resize_factor=None):
    """Returns (xml_string, meta). meta carries what the env layer needs beyond the XML:
    part names in XML document order, *_initpos numerics, horizontal radii, robot/gripper joint names."""
    assets_root = assets_root or default_assets_root()
    if assets_root is None:
        raise FileNotFoundError("furniture assets not found; set FURNITURE_ASSETS or use a compiled model (.npz)")
    world = ET.parse(os.path.join(assets_root, "base.xml")).getroot()

    # arena: furniture.py:1967-1977 + arena.py:86-103
    arena = ET.parse(os.path.join(assets_root, "arenas", "floor_arena.xml")).getroot()
    floor = arena.find("./worldbody/geom[@name='FLOOR']")
    floor_half = np.array([1.5, 1.0, 0.125]) / 2
    floor.set("size", " ".join(str(x) for x in floor_half))
    floor.set("friction", "2.0 0.005 0.0001")
    _merge(world, arena)

    meta = {"agent": agent, "furniture": furniture}
    if agent == "Sawyer":
        rxml = "robots/sawyer/robot_torque.xml" if use_torque else "robots/sawyer/robot.xml"
        robot = ET.parse(os.path.join(assets_root, rxml)).getroot()
        gripper = ET.parse(os.path.join(assets_root, "grippers", "two_finger_gripper.xml")).getroot()
        hand = robot.find("./worldbody//body[@name='right_hand']")
        for body in list(_section(gripper, "worldbody")):
            hand.append(body)
        _merge(robot, gripper, merge_body=False)
        base = robot.find("./worldbody/body[@name='base']")
        pos = np.array([0, 0.65, -0.7]) - SAWYER_BOTTOM_OFFSET  # furniture.py:1901, sawyer_robot.py:24-29
        base.set("pos", " ".join(str(x) for x in pos))
        base.set("quat", "1 0 0 -1")  # furniture.py:1902 (un-normalised; the compiler normalises)
        _merge(world, robot)
        meta["robot_joints"] = ["right_j%d" % i for i in range(7)]
        meta["gripper_joints"] = ["r_gripper_l_finger_joint", "r_gripper_r_finger_joint"]
        meta["robot_init_qpos"] = SAWYER_INIT_QPOS.copy()
        meta["gripper_init_qpos"] = GRIPPER_INIT_QPOS.copy()
        meta["l_finger_geoms"] = ["l_finger_g0", "l_finger_g1", "l_fingertip_g0"]
        meta["r_finger_geoms"] = ["r_finger_g0", "r_finger_g1", "r_fingertip_g0"]
        # Robot.is_robot_part: sawyer_robot.py:117-141 + two_finger_gripper.py:41-51
        meta["robot_contact_geoms"] = (
            ["pedestal_collision", "right_arm_base_link_collision", "right_l0_collision", "head_collision", "screen_collision"]
            + ["right_l%d_collision" % i for i in range(1, 7)]
            + ["right_l4_2_collision", "right_l2_2_collision", "right_l1_2_collision"]
            + ["r_finger_g0", "r_finger_g1", "l_finger_g0", "l_finger_g1", "r_fingertip_g0", "l_fingertip_g0", "right_gripper_base_collision"]
        )
        meta["eef_site"] = "grip_site"
        meta["hand_body"] = "right_hand"
    elif agent == "Baxter":
        # furniture.py:1925-1939 + baxter_robot.py + two_finger_gripper.py: right gripper on right_hand, left gripper on left_hand
        robot = ET.parse(os.path.join(assets_root, "robots/baxter/robot_torque.xml" if use_torque else "robots/baxter/robot.xml")).getroot()
        for a in _section(robot, "asset"):  # mesh files of the robot are relative to its own directory
            if a.get("file") is not None:
                a.set("file", os.path.join(assets_root, "robots", "baxter", a.get("file")))
        for hand_name, gx in (("right_hand", "two_finger_gripper.xml"), ("left_hand", "left_two_finger_gripper.xml")):
            gripper = ET.parse(os.path.join(assets_root, "grippers", gx)).getroot()
            hand = robot.find("./worldbody//body[@name='%s']" % hand_name)
            for body in list(_section(gripper, "worldbody")):
                hand.append(body)
            _merge(robot, gripper, merge_body=False)
        base = robot.find("./worldbody/body[@name='base']")
        pos = np.array([0, 0.65, -0.7]) - BAXTER_BOTTOM_OFFSET
        base.set("pos", " ".join(str(x) for x in pos))
        base.set("quat", "1 0 0 -1")
        _merge(world, robot)
        arm_j = ["s0", "s1", "e0", "e1", "w0", "w1", "w2"]
        meta["robot_joints"] = ["right_" + a for a in arm_j] + ["left_" + a for a in arm_j]  # baxter_robot.py:38-42
        meta["gripper_joints"] = ["r_gripper_l_finger_joint", "r_gripper_r_finger_joint", "l_gripper_l_finger_joint", "l_gripper_r_finger_joint"]
        meta["robot_init_qpos"] = BAXTER_INIT_QPOS.copy()
        meta["gripper_init_qpos"] = np.concatenate([GRIPPER_INIT_QPOS, GRIPPER_INIT_QPOS])
        meta["l_finger_geoms"] = ["l_finger_g0", "l_finger_g1", "l_fingertip_g0"]          # arm "right"
        meta["r_finger_geoms"] = ["r_finger_g0", "r_finger_g1", "r_fingertip_g0"]
        meta["l_finger_geoms2"] = ["l_g_l_finger_g0", "l_g_l_finger_g1", "l_g_l_fingertip_g0"]  # arm "left"
        meta["r_finger_geoms2"] = ["l_g_r_finger_g0", "l_g_r_finger_g1", "l_g_r_fingertip_g0"]
        meta["robot_contact_geoms"] = (  # baxter_robot.py:71-86 + both grippers' contact_geoms
            ["right_%s_collision" % n for n in ("upper_shoulder", "lower_shoulder", "upper_elbow", "lower_elbow", "upper_forearm", "lower_forearm", "wrist")]
            + ["left_%s_collision" % n for n in ("upper_shoulder", "lower_shoulder", "upper_elbow", "lower_elbow", "upper_forearm", "lower_forearm")]
            + ["r_finger_g0", "r_finger_g1", "l_finger_g0", "l_finger_g1", "r_fingertip_g0", "l_fingertip_g0", "right_gripper_base_collision"]
            + ["l_g_r_finger_g0", "l_g_r_finger_g1", "l_g_l_finger_g0", "l_g_l_finger_g1", "l_g_r_fingertip_g0", "l_g_l_fingertip_g0", "left_gripper_base_collision"]
        )
        meta["eef_site"], meta["hand_body"] = "grip_site", "right_hand"
        meta["eef_site2"], meta["hand_body2"] = "l_g_grip_site", "left_hand"
    elif agent == "Cursor":
        # furniture.py:1949-1954 + robots/cursor.py: two static cursor boxes, half size = margin = move_speed / 2 (default 0.1 / 2), gap 10
        robot = ET.parse(os.path.join(assets_root, "robots", "cursor", "robot.xml")).getroot()
        half = 0.05
        for nm in ("cursor0", "cursor1"):
            robot.find("./worldbody/body[@name='%s']" % nm).set("pos", "0 0 %s" % half)
            g = robot.find("./worldbody/body/geom[@name='%s']" % nm)
            g.set("size", "%s %s %s" % (half, half, half))
            g.set("margin", str(half))
        _merge(world, robot)
        meta.update(robot_joints=[], gripper_joints=[], robot_init_qpos=np.zeros(0), gripper_init_qpos=np.zeros(0),
                    l_finger_geoms=["cursor0"], r_finger_geoms=["cursor1"],  # touch bit 0 / 1 of a part = cursor0 / cursor1 on it
                    robot_contact_geoms=["cursor0", "cursor1"], movable_geoms=["cursor0", "cursor1"], eef_site=None, hand_body=None)
    elif agent == "None":
        meta.update(robot_joints=[], gripper_joints=[], robot_init_qpos=np.zeros(0), gripper_init_qpos=np.zeros(0),
                    l_finger_geoms=[], r_finger_geoms=[], robot_contact_geoms=[], eef_site=None, hand_body=None)
    else:
        raise NotImplementedError("agent %s: Sawyer, Baxter, Cursor and None are composed" % agent)

    # furniture parts: furniture.py:1979-2001 + floor_task.py:55-72 + objects.py:186-206
    obj = ET.parse(os.path.join(assets_root, "objects", furniture + ".xml")).getroot()
    if resize_factor:  # furn_size_rand / manual resize: furniture.py:1985-1992
        _rescale_objects(obj, float(resize_factor))
        meta["resize_factor"] = float(resize_factor)
    part_names = [b.get("name") for b in obj.iter("body")]  # base.py:159-167 (root.iter => document order)
    dst_asset = _section(world, "asset")
    for a in list(_section(obj, "asset")):
        if a.get("file") is not None:  # MujocoXML.resolve_asset_dependency, models/base.py:55-62
            a.set("file", os.path.join(assets_root, "objects", a.get("file")))
        nm = a.get("name")
        if nm is None or dst_asset.find("./{}[@name='{}']".format(a.tag, nm)) is None:
            dst_asset.append(a)
    init_qpos = {}
    custom = obj.find("custom")
    if custom is not None:  # objects.py:149-164
        for num in custom:
            nm = num.get("name", "")
            if "initpos" in nm:
                key = "_".join(nm.split("_")[0:-1])
                if key in part_names:
                    init_qpos[key] = _floats(num.get("data"))
    radii = {}
    for name in part_names:
        body = copy.deepcopy(obj.find("./worldbody/body[@name='%s']" % name))
        geoms = body.findall("geom")
        for i, g in enumerate(geoms):
            gname = g.get("name")
            if not (gname.startswith("noviz") or gname.startswith("collision")):
                g.set("name", "{}-{}".format(name, i))
            g.set("friction", "1 10 0.5")
        ET.SubElement(body, "site", {"pos": "0 0 0", "size": "0.002 0.002 0.002", "rgba": "1 0 0 0", "type": "sphere", "name": name})
        ET.SubElement(body, "joint", {"name": name, "type": "free", "damping": "0.0001"})
        _section(world, "worldbody").append(body)
        hs = obj.find("./worldbody/body/site[@name='%s_horizontal_radius_site']" % name)
        radii[name] = float(hs.get("size")) if hs is not None else 0.0
    for eq in list(_section(obj, "equality")):
        _section(world, "equality").append(eq)
    meta["part_names"] = part_names
    recipe = load_recipe(furniture, assets_root)
    if recipe is not None:
        import json

        meta["recipe_json"] = json.dumps(recipe)
    init_qpos.update(place_unlisted_parts(part_names, init_qpos, radii, placement_seed))
    meta["part_init_qpos"] = init_qpos
    meta["part_radius"] = radii
    with io.StringIO() as s:
        s.write(ET.tostring(world, encoding="unicode"))
        return s.getvalue(), meta


# --------------------------------------------------------------------------------------
# compiled model
# --------------------------------------------------------------------------------------


@dataclass
class Model:
    """Flat tables of one compiled scene (MuJoCo-style names). All float arrays are float64 here;
    the engine down-converts what it needs to fp32."""

    a: dict = field(default_factory=dict)  # name -> ndarray / scalar
    names: dict = field(default_factory=dict)  # 'body'|'jnt'|'geom'|'site'|'actuator'|'eq' -> list[str]
    meta: dict = field(default_factory=dict)

    def __getattr__(self, k):
        a = object.__getattribute__(self, "a")
        if k in a:
            return a[k]
        raise AttributeError(k)

    def name2id(self, kind, name):
        return self.names[kind].index(name)

    def save(self, path):
        import json

        meta = {}
        for k, v in self.meta.items():
            if isinstance(v, np.ndarray):
                meta[k] = {"__nd__": v.tolist()}
            elif isinstance(v, dict):
                meta[k] = {kk: (vv.tolist() if isinstance(vv, np.ndarray) else vv) for kk, vv in v.items()}
            else:
                meta[k] = v
        np.savez_compressed(path, __names__=json.dumps(self.names), __meta__=json.dumps(meta), **{k: np.asarray(v) for k, v in self.a.items()})

    @staticmethod
    def load(path):
        import json

        z = np.load(path, allow_pickle=False)
        m = Model()
        for k in z.files:
            if k == "__names__":
                m.names = json.loads(str(z[k]))
            elif k == "__meta__":
                meta = json.loads(str(z[k]))
                for kk, vv in meta.items():
                    if isinstance(vv, dict) and "__nd__" in vv:
                        meta[kk] = np.array(vv["__nd__"])
                    elif isinstance(vv, dict):
                        meta[kk] = {a: (np.array(b) if isinstance(b, list) and b and isinstance(b[0], float) else b) for a, b in vv.items()}
                m.meta = meta
            else:
                v = z[k]
                m.a[k] = v.item() if v.shape == () else v
        return m


class _Defaults:
    """<default> classes: nested <default class="x"> inherit from the enclosing one."""

    def __init__(self, root):
        self.cls = {"main": {}}
        for d in root.findall("default"):
            self._walk(d, "main", top=True)

    def _walk(self, node, parent, top=False):
        name = node.get("class") or ("main" if top else None)
        if name is None:
            name = parent
        if name not in self.cls:
            self.cls[name] = copy.deepcopy(self.cls[parent])
        for child in node:
            if child.tag == "default":
                self._walk(child, name)
            else:
                self.cls[name].setdefault(child.tag, {}).update(child.attrib)

    def get(self, tag, el, childclass):
        c = el.get("class") or childclass or "main"
        out = dict(self.cls.get(c, self.cls["main"]).get(tag, {}))
        out.update(el.attrib)
        return out


def _orient(attr):
    if "quat" in attr:
        return q_norm(_floats(attr["quat"]))
    if "euler" in attr:
        return q_norm(euler_xyz_to_q(_floats(attr["euler"])))
    if "axisangle" in attr:
        v = _floats(attr["axisangle"])
        return q_norm(q_axis_angle(v[:3] / np.linalg.norm(v[:3]), v[3]))
    return np.array([1.0, 0.0, 0.0, 0.0])


def _geom_mass_inertia(gtype, size, density):
    """mass and principal inertia (geom frame, about geom centre) of a primitive."""
    if gtype == GEOM_BOX:
        a, b, c = size
        m = density * 8 * a * b * c
        I = np.array([b * b + c * c, a * a + c * c, a * a + b * b]) * m / 3.0
    elif gtype == GEOM_SPHERE:
        r = size[0]
        m = density * 4.0 / 3.0 * math.pi * r**3
        I = np.full(3, 0.4 * m * r * r)
    elif gtype == GEOM_CYLINDER:
        r, h = size[0], size[1]
        m = density * math.pi * r * r * 2 * h
        I = np.array([m * (3 * r * r + 4 * h * h) / 12.0] * 2 + [m * r * r / 2.0])
    elif gtype == GEOM_CAPSULE:
        r, h = size[0], size[1]
        mc = density * math.pi * r * r * 2 * h
        ms = density * 4.0 / 3.0 * math.pi * r**3
        m = mc + ms
        Iz = mc * r * r / 2 + ms * 0.4 * r * r
        Ix = mc * (3 * r * r + 4 * h * h) / 12.0 + ms * (0.4 * r * r + h * h + 0.75 * r * h)
        I = np.array([Ix, Ix, Iz])
    else:
        m, I = 0.0, np.zeros(3)
    return m, I


def load_stl(path):
    """triangles (n, 3, 3) of a binary STL (the furniture meshes are Rhino binary exports)"""
    raw = open(path, "rb").read()
    n = int(np.frombuffer(raw[80:84], dtype="<u4")[0])
    if len(raw) != 84 + 50 * n:
        raise NotImplementedError("not a binary STL: " + path)
    rec = np.frombuffer(raw[84:], dtype=np.dtype([("n", "<f4", 3), ("v", "<f4", (3, 3)), ("a", "<u2")]), count=n)
    return rec["v"].astype(np.float64)


def mesh_mass_properties(tri, density):
    """mass, centre of mass and inertia tensor about it (mesh frame) of the solid bounded by a closed triangle mesh: exact
    volume integrals over the signed tetrahedra (origin, v0, v1, v2).  MuJoCo 2.0 sums pyramids from the faces to the
    mesh centroid, which is the same number for the closed, consistently oriented meshes shipped with the furniture."""
    a, b, c = tri[:, 0], tri[:, 1], tri[:, 2]
    vol6 = np.einsum("ij,ij->i", a, np.cross(b, c))  # 6 x signed volume
    V = vol6.sum() / 6.0
    sgn = 1.0 if V >= 0 else -1.0
    com = (vol6[:, None] * (a + b + c)).sum(0) / (24.0 * V)
    # second moment: for a tetrahedron (0, a, b, c), integral of x x^T dV = det / 120 * (s s^T + a a^T + b b^T + c c^T), s = a + b + c
    sm = a + b + c
    S = sum(np.einsum("i,ij,ik->jk", vol6, u, u) for u in (sm, a, b, c)) / 120.0
    mass = density * abs(V)
    S = S * sgn * density                       # density-weighted second moment about the origin
    S -= mass * np.outer(com, com)              # ... about the centre of mass
    I = np.trace(S) * np.eye(3) - S
    return mass, com, I


def compile_mjcf(xml_string, meta=None):
    root = ET.fromstring(xml_string)
    comp = root.find("compiler")
    angle_rad = comp is not None and comp.get("angle") == "radian"
    ang = 1.0 if angle_rad else math.pi / 180.0
    opt = root.find("option")
    oa = opt.attrib if opt is not None else {}
    timestep = float(oa.get("timestep", 0.002))
    gravity = _floats(oa.get("gravity"), 3, [0, 0, -9.81])
    impratio = float(oa.get("impratio", 1.0))
    cone_elliptic = 1 if oa.get("cone", "pyramidal") == "elliptic" else 0
    tolerance = float(oa.get("tolerance", 1e-8))
    iterations = int(oa.get("iterations", 100))
    dfl = _Defaults(root)

    B = dict(parent=[], pos=[], quat=[], ipos=[], iquat=[], mass=[], inertia=[], name=[], explicit=[])
    J = dict(type=[], body=[], pos=[], axis=[], limited=[], range=[], damping=[], name=[], solref=[], solimp=[], armature=[])
    G = dict(type=[], body=[], pos=[], quat=[], size=[], contype=[], conaffinity=[], condim=[], friction=[], solref=[], solimp=[], margin=[], gap=[], name=[], density=[],
             meshadr=[], meshnum=[])
    mesh_verts = []  # convex-hull vertices of the mesh colliders, geom frame (one block per mesh geom)
    S = dict(body=[], pos=[], quat=[], name=[])
    meshes = {}
    asset = root.find("asset")
    if asset is not None:
        for me in asset.findall("mesh"):
            nm = me.get("name") or os.path.splitext(os.path.basename(me.get("file", "")))[0]
            meshes[nm] = dict(file=me.get("file"), scale=_floats(me.get("scale"), 3, [1, 1, 1]))
    mesh_inertia = {}  # body id -> [(mass, com in the body frame, inertia about it in the body frame)] of non-colliding mesh geoms

    def add_body(el, parent, childclass):
        attr = el.attrib
        bid = len(B["parent"])
        B["parent"].append(parent)
        B["name"].append(attr.get("name", "world" if parent < 0 else "body%d" % bid))
        B["pos"].append(_floats(attr.get("pos"), 3, [0, 0, 0]))
        B["quat"].append(_orient(attr))
        cc = attr.get("childclass") or childclass
        inert = el.find("inertial")
        if inert is not None:
            ia = inert.attrib
            B["explicit"].append(True)
            B["ipos"].append(_floats(ia.get("pos"), 3, [0, 0, 0]))
            B["iquat"].append(_orient(ia))
            B["mass"].append(float(ia.get("mass", 0)))
            if "diaginertia" in ia:
                B["inertia"].append(_floats(ia["diaginertia"]))
            elif "fullinertia" in ia:
                f = _floats(ia["fullinertia"])
                M = np.array([[f[0], f[3], f[4]], [f[3], f[1], f[5]], [f[4], f[5], f[2]]])
                w, V = np.linalg.eigh(M)
                if np.linalg.det(V) < 0:
                    V[:, 2] *= -1
                B["inertia"].append(w)
                B["iquat"][-1] = mat_to_q(V)
            else:
                B["inertia"].append(np.zeros(3))
        else:
            B["explicit"].append(False)
            B["ipos"].append(np.zeros(3))
            B["iquat"].append(np.array([1.0, 0, 0, 0]))
            B["mass"].append(0.0)
            B["inertia"].append(np.zeros(3))
        for child in el:
            if child.tag == "joint" or child.tag == "freejoint":
                a = dfl.get("joint", child, cc)
                jt = "free" if child.tag == "freejoint" else a.get("type", "hinge")
                J["type"].append({"free": JNT_FREE, "slide": JNT_SLIDE, "hinge": JNT_HINGE}[jt])
                J["body"].append(bid)
                J["name"].append(a.get("name", "jnt%d" % len(J["name"])))
                J["pos"].append(_floats(a.get("pos"), 3, [0, 0, 0]))
                ax = _floats(a.get("axis"), 3, [0, 0, 1])
                J["axis"].append(ax / max(np.linalg.norm(ax), 1e-14))
                J["limited"].append(1 if a.get("limited", "false") == "true" else 0)
                rng = _floats(a.get("range"), 2, [0, 0])
                if jt == "hinge":
                    rng = rng * ang
                J["range"].append(rng)
                J["damping"].append(float(a.get("damping", 0)))
                J["armature"].append(float(a.get("armature", 0)))
                J["solref"].append(_floats(a.get("solreflimit"), 2, [0.02, 1]))
                J["solimp"].append(_floats(a.get("solimplimit"), 5, [0.9, 0.95, 0.001, 0.5, 2]))
            elif child.tag == "geom":
                a = dfl.get("geom", child, cc)
                tname = a.get("type", "sphere")
                contype = int(a.get("contype", 1))
                conaff = int(a.get("conaffinity", 1))
                density = float(a.get("density", 1000))
                if tname == "mesh":
                    # visual meshes carry contype=conaffinity=0; with density 0 they are ignored (A.1), with a density they still
                    # add their mass and inertia to the body (4 furniture models).  Mesh *colliders* (3 furniture models) collide
                    # through the convex hull of their vertices, as in MuJoCo (mesh geoms are convexified for collision).
                    mesh = meshes.get(a.get("mesh"))
                    collider = contype != 0 or conaff != 0
                    tri = None
                    if mesh is not None and ((density != 0 and inert is None) or collider):
                        tri = load_stl(mesh["file"]) * mesh["scale"]
                    elif (density != 0 and inert is None) or collider:
                        raise NotImplementedError("mesh asset '%s' of geom '%s' not found" % (a.get("mesh"), a.get("name")))
                    if density != 0 and inert is None:
                        m_, c_, I_ = mesh_mass_properties(tri, density)
                        Rg = q_to_mat(_orient(a))
                        mesh_inertia.setdefault(bid, []).append((m_, _floats(a.get("pos"), 3, [0, 0, 0]) + Rg @ c_, Rg @ I_ @ Rg.T))
                    if not collider:
                        continue
                    try:
                        from scipy.spatial import ConvexHull
                    except Exception as e:  # pragma: no cover
                        raise NotImplementedError("mesh collider geom '%s' needs scipy for its convex hull (%s)" % (a.get("name"), e))
                    verts = np.unique(tri.reshape(-1, 3), axis=0)
                    hv = verts[np.sort(ConvexHull(verts).vertices)]
                    lo, hi = hv.min(0), hv.max(0)
                    G["type"].append(GEOM_MESH)
                    G["body"].append(bid)
                    G["name"].append(a.get("name", ""))
                    G["pos"].append(_floats(a.get("pos"), 3, [0, 0, 0]))
                    G["quat"].append(_orient(a))
                    G["size"].append(0.5 * (hi - lo))  # half extents of the hull's bounding box (informative; collision uses the vertices)
                    G["contype"].append(contype)
                    G["conaffinity"].append(conaff)
                    G["condim"].append(int(a.get("condim", 3)))
                    G["friction"].append(_floats(a.get("friction"), 3, [1, 0.005, 0.0001]))
                    G["solref"].append(_floats(a.get("solref"), 2, [0.02, 1]))
                    G["solimp"].append(_floats(a.get("solimp"), 5, [0.9, 0.95, 0.001, 0.5, 2]))
                    G["margin"].append(float(a.get("margin", 0)))
                    G["gap"].append(float(a.get("gap", 0)))
                    G["density"].append(0.0)  # mass already taken from the triangle mesh above
                    G["meshadr"].append(sum(len(v) for v in mesh_verts))
                    G["meshnum"].append(len(hv))
                    mesh_verts.append(hv)
                    continue
                if tname not in GEOM_TYPES:
                    raise NotImplementedError("geom type " + tname)
                size = _floats(a.get("size"), 3, [0, 0, 0])
                G["type"].append(GEOM_TYPES[tname])
                G["body"].append(bid)
                G["name"].append(a.get("name", ""))
                G["pos"].append(_floats(a.get("pos"), 3, [0, 0, 0]))
                G["quat"].append(_orient(a))
                G["size"].append(size)
                G["contype"].append(contype)
                G["conaffinity"].append(conaff)
                G["condim"].append(int(a.get("condim", 3)))
                G["friction"].append(_floats(a.get("friction"), 3, [1, 0.005, 0.0001]))
                G["solref"].append(_floats(a.get("solref"), 2, [0.02, 1]))
                G["solimp"].append(_floats(a.get("solimp"), 5, [0.9, 0.95, 0.001, 0.5, 2]))
                G["margin"].append(float(a.get("margin", 0)))
                G["gap"].append(float(a.get("gap", 0)))
                G["density"].append(density)
                G["meshadr"].append(-1)
                G["meshnum"].append(0)
            elif child.tag == "site":
                a = dfl.get("site", child, cc)
                S["body"].append(bid)
                S["name"].append(a.get("name", "site%d" % len(S["name"])))
                S["pos"].append(_floats(a.get("pos"), 3, [0, 0, 0]))
                S["quat"].append(_orient(a))
        for child in el:
            if child.tag == "body":
                add_body(child, bid, cc)

    wb = root.find("worldbody")
    wb_attr = dict(wb.attrib)
    wb.attrib.clear()
    wb.set("name", "world")
    add_body(wb, -1, None)
    wb.attrib.clear()
    wb.attrib.update(wb_attr)
    nbody = len(B["parent"])
    B["parent"][0] = 0

    # MuJoCo groups geoms / sites / joints by body id (ids follow body order)
    def regroup(T):
        order = sorted(range(len(T["body"])), key=lambda i: (T["body"][i], i))
        for k in T:
            T[k] = [T[k][i] for i in order]

    regroup(G)
    regroup(S)
    regroup(J)
    ngeom, nsite, njnt = len(G["body"]), len(S["body"]), len(J["body"])

    # inertia from geoms for bodies without <inertial>
    for b in range(nbody):
        if B["explicit"][b]:
            continue
        gs = [i for i in range(ngeom) if G["body"][i] == b and G["density"][i] > 0 and G["type"][i] not in (GEOM_PLANE, GEOM_MESH)]
        if not gs and b not in mesh_inertia:
            continue
        ms, cs, Is = [], [], []
        for i in gs:
            m, I = _geom_mass_inertia(G["type"][i], G["size"][i], G["density"][i])
            R = q_to_mat(G["quat"][i])
            ms.append(m)
            cs.append(G["pos"][i])
            Is.append(R @ np.diag(I) @ R.T)
        for m, c, I in mesh_inertia.get(b, []):
            ms.append(m)
            cs.append(np.asarray(c, dtype=np.float64))
            Is.append(I)
        M = sum(ms)
        if M <= 0:
            continue
        com = sum(m * c for m, c in zip(ms, cs)) / M
        Itot = np.zeros((3, 3))
        for m, c, I in zip(ms, cs, Is):
            d = c - com
            Itot += I + m * (d @ d * np.eye(3) - np.outer(d, d))
        w, V = np.linalg.eigh(Itot)
        if np.linalg.det(V) < 0:
            V[:, 2] *= -1
        B["mass"][b] = M
        B["ipos"][b] = com
        B["iquat"][b] = mat_to_q(V)
        B["inertia"][b] = w

    # joints -> qpos / dof addressing
    jnt_qposadr, jnt_dofadr = [], []
    nq = nv = 0
    for j in range(njnt):
        jnt_qposadr.append(nq)
        jnt_dofadr.append(nv)
        if J["type"][j] == JNT_FREE:
            nq += 7
            nv += 6
        else:
            nq += 1
            nv += 1
    body_jntadr = [-1] * nbody
    body_jntnum = [0] * nbody
    for j in range(njnt):
        b = J["body"][j]
        if body_jntadr[b] < 0:
            body_jntadr[b] = j
        body_jntnum[b] += 1
    body_dofadr = [-1] * nbody
    body_dofnum = [0] * nbody
    dof_bodyid, dof_jntid, dof_damping, dof_armature = [], [], [], []
    for j in range(njnt):
        n = 6 if J["type"][j] == JNT_FREE else 1
        b = J["body"][j]
        if body_dofadr[b] < 0:
            body_dofadr[b] = jnt_dofadr[j]
        body_dofnum[b] += n
        for _ in range(n):
            dof_bodyid.append(b)
            dof_jntid.append(j)
            dof_damping.append(J["damping"][j])
            dof_armature.append(J["armature"][j])
    # weld id (nearest ancestor-or-self with a joint; 0 = welded to world) and tree root
    body_weldid = [0] * nbody
    body_rootid = [0] * nbody
    for b in range(1, nbody):
        p = B["parent"][b]
        body_weldid[b] = b if body_jntnum[b] > 0 else body_weldid[p]
        body_rootid[b] = b if p == 0 else body_rootid[p]
    # dof parent (previous dof up the kinematic chain)
    dof_parentid = [-1] * nv
    last_dof_of_body = [-1] * nbody
    for b in range(1, nbody):
        p = B["parent"][b]
        prev = last_dof_of_body[p]
        if body_dofnum[b] > 0:
            for k in range(body_dofnum[b]):
                d = body_dofadr[b] + k
                dof_parentid[d] = prev
                prev = d
        last_dof_of_body[b] = prev
    qpos0 = np.zeros(nq)
    for j in range(njnt):
        if J["type"][j] == JNT_FREE:
            b = J["body"][j]
            qpos0[jnt_qposadr[j] : jnt_qposadr[j] + 3] = B["pos"][b]
            qpos0[jnt_qposadr[j] + 3 : jnt_qposadr[j] + 7] = B["quat"][b]

    # actuators
    act = root.find("actuator")
    A = dict(type=[], jnt=[], gain=[], bias=[], ctrllimited=[], ctrlrange=[], forcelimited=[], forcerange=[], name=[], gear=[])
    if act is not None:
        for el in act:
            a = dfl.get(el.tag, el, None)
            if el.tag not in ("motor", "position", "velocity"):
                raise NotImplementedError("actuator " + el.tag)
            A["name"].append(a.get("name", ""))
            A["jnt"].append(J["name"].index(a["joint"]))
            A["gear"].append(_floats(a.get("gear"), 1, [1.0])[0])
            A["ctrllimited"].append(1 if a.get("ctrllimited", "false") == "true" else 0)
            A["ctrlrange"].append(_floats(a.get("ctrlrange"), 2, [0, 0]))
            A["forcelimited"].append(1 if a.get("forcelimited", "false") == "true" else 0)
            A["forcerange"].append(_floats(a.get("forcerange"), 2, [0, 0]))
            if el.tag == "motor":
                A["type"].append(ACT_MOTOR)
                A["gain"].append(1.0)
                A["bias"].append(np.zeros(3))
            elif el.tag == "position":
                kp = float(a.get("kp", 1))
                A["type"].append(ACT_POSITION)
                A["gain"].append(kp)
                A["bias"].append(np.array([0, -kp, 0.0]))
            else:
                kv = float(a.get("kv", 1))
                A["type"].append(ACT_VELOCITY)
                A["gain"].append(kv)
                A["bias"].append(np.array([0, 0.0, -kv]))
    nu = len(A["type"])

    # equalities (weld only)
    E = dict(b1=[], b2=[], active=[], data=[], solref=[], solimp=[])
    eqs = root.find("equality")
    if eqs is not None:
        for el in eqs:
            if el.tag != "weld":
                raise NotImplementedError("equality " + el.tag)
            a = dfl.get("weld", el, None)
            E["b1"].append(B["name"].index(a["body1"]))
            E["b2"].append(B["name"].index(a["body2"]) if "body2" in a else 0)
            E["active"].append(0 if a.get("active", "true") == "false" else 1)
            E["solref"].append(_floats(a.get("solref"), 2, [0.02, 1]))
            E["solimp"].append(_floats(a.get("solimp"), 5, [0.9, 0.95, 0.001, 0.5, 2]))
            E["data"].append(None)
    neq = len(E["b1"])

    # contact excludes
    excl = []
    con = root.find("contact")
    if con is not None:
        for el in con:
            if el.tag == "exclude":
                excl.append((B["name"].index(el.get("body1")), B["name"].index(el.get("body2"))))
            else:
                raise NotImplementedError("contact/" + el.tag)

    a = {}
    a["nq"], a["nv"], a["nu"], a["nbody"], a["njnt"], a["ngeom"], a["nsite"], a["neq"] = nq, nv, nu, nbody, njnt, ngeom, nsite, neq
    a["opt_timestep"], a["opt_gravity"], a["opt_impratio"], a["opt_cone_elliptic"] = timestep, gravity, impratio, cone_elliptic
    a["opt_tolerance"], a["opt_iterations"] = tolerance, iterations
    a["body_parentid"] = np.array(B["parent"], dtype=np.int32)
    a["body_weldid"] = np.array(body_weldid, dtype=np.int32)
    a["body_rootid"] = np.array(body_rootid, dtype=np.int32)
    a["body_jntadr"] = np.array(body_jntadr, dtype=np.int32)
    a["body_jntnum"] = np.array(body_jntnum, dtype=np.int32)
    a["body_dofadr"] = np.array(body_dofadr, dtype=np.int32)
    a["body_dofnum"] = np.array(body_dofnum, dtype=np.int32)
    a["body_pos"] = np.array(B["pos"]).reshape(nbody, 3)
    a["body_quat"] = np.array(B["quat"]).reshape(nbody, 4)
    a["body_ipos"] = np.array(B["ipos"]).reshape(nbody, 3)
    a["body_iquat"] = np.array(B["iquat"]).reshape(nbody, 4)
    a["body_mass"] = np.array(B["mass"], dtype=np.float64)
    a["body_inertia"] = np.array(B["inertia"]).reshape(nbody, 3)
    a["jnt_type"] = np.array(J["type"], dtype=np.int32)
    a["jnt_bodyid"] = np.array(J["body"], dtype=np.int32)
    a["jnt_qposadr"] = np.array(jnt_qposadr, dtype=np.int32)
    a["jnt_dofadr"] = np.array(jnt_dofadr, dtype=np.int32)
    a["jnt_pos"] = np.array(J["pos"]).reshape(njnt, 3)
    a["jnt_axis"] = np.array(J["axis"]).reshape(njnt, 3)
    a["jnt_limited"] = np.array(J["limited"], dtype=np.int32)
    a["jnt_range"] = np.array(J["range"]).reshape(njnt, 2)
    a["jnt_solref"] = np.array(J["solref"]).reshape(njnt, 2)
    a["jnt_solimp"] = np.array(J["solimp"]).reshape(njnt, 5)
    a["dof_bodyid"] = np.array(dof_bodyid, dtype=np.int32)
    a["dof_jntid"] = np.array(dof_jntid, dtype=np.int32)
    a["dof_parentid"] = np.array(dof_parentid, dtype=np.int32)
    a["dof_damping"] = np.array(dof_damping, dtype=np.float64)
    a["dof_armature"] = np.array(dof_armature, dtype=np.float64)
    a["qpos0"] = qpos0
    a["geom_type"] = np.array(G["type"], dtype=np.int32)
    a["geom_bodyid"] = np.array(G["body"], dtype=np.int32)
    a["geom_contype"] = np.array(G["contype"], dtype=np.int32)
    a["geom_conaffinity"] = np.array(G["conaffinity"], dtype=np.int32)
    a["geom_condim"] = np.array(G["condim"], dtype=np.int32)
    a["geom_size"] = np.array(G["size"]).reshape(ngeom, 3)
    a["geom_pos"] = np.array(G["pos"]).reshape(ngeom, 3)
    a["geom_quat"] = np.array(G["quat"]).reshape(ngeom, 4)
    a["geom_friction"] = np.array(G["friction"]).reshape(ngeom, 3)
    a["geom_solref"] = np.array(G["solref"]).reshape(ngeom, 2)
    a["geom_solimp"] = np.array(G["solimp"]).reshape(ngeom, 5)
    a["geom_margin"] = np.array(G["margin"], dtype=np.float64)
    a["geom_gap"] = np.array(G["gap"], dtype=np.float64)
    rb = np.zeros(ngeom)
    mesh_verts_all = np.concatenate(mesh_verts, 0) if mesh_verts else np.zeros((0, 3))
    for i in range(ngeom):
        t, s = G["type"][i], G["size"][i]
        if t == GEOM_MESH:
            rb[i] = float(np.linalg.norm(mesh_verts_all[G["meshadr"][i] : G["meshadr"][i] + G["meshnum"][i]], axis=1).max())
        else:
            rb[i] = {GEOM_PLANE: 0.0, GEOM_SPHERE: s[0], GEOM_CAPSULE: s[0] + s[1], GEOM_CYLINDER: math.hypot(s[0], s[1]), GEOM_BOX: float(np.linalg.norm(s))}[t]
    a["geom_rbound"] = rb
    a["geom_meshadr"] = np.array(G["meshadr"], dtype=np.int32)
    a["geom_meshnum"] = np.array(G["meshnum"], dtype=np.int32)
    a["mesh_vert"] = mesh_verts_all
    a["site_bodyid"] = np.array(S["body"], dtype=np.int32)
    a["site_pos"] = np.array(S["pos"]).reshape(nsite, 3)
    a["site_quat"] = np.array(S["quat"]).reshape(nsite, 4)
    a["actuator_type"] = np.array(A["type"], dtype=np.int32)
    a["actuator_jntid"] = np.array(A["jnt"], dtype=np.int32)
    a["actuator_gear"] = np.array(A["gear"], dtype=np.float64)
    a["actuator_gainprm"] = np.array(A["gain"], dtype=np.float64)
    a["actuator_biasprm"] = np.array(A["bias"]).reshape(nu, 3)
    a["actuator_ctrllimited"] = np.array(A["ctrllimited"], dtype=np.int32)
    a["actuator_ctrlrange"] = np.array(A["ctrlrange"]).reshape(nu, 2)
    a["actuator_forcelimited"] = np.array(A["forcelimited"], dtype=np.int32)
    a["actuator_forcerange"] = np.array(A["forcerange"]).reshape(nu, 2)
    a["eq_obj1id"] = np.array(E["b1"], dtype=np.int32)
    a["eq_obj2id"] = np.array(E["b2"], dtype=np.int32)
    a["eq_active"] = np.array(E["active"], dtype=np.int32)
    a["eq_solref"] = np.array(E["solref"]).reshape(neq, 2)
    a["eq_solimp"] = np.array(E["solimp"]).reshape(neq, 5)
    a["exclude"] = np.array(excl, dtype=np.int32).reshape(len(excl), 2)

    m = Model(a=a, names=dict(body=B["name"], jnt=J["name"], geom=G["name"], site=S["name"], actuator=A["name"]), meta=meta or {})
    _set_const(m)
    # weld relpose at qpos0: body2 pose in body1 frame (the compiler default when relpose is unspecified)
    kin = kinematics_np(m, m.qpos0)
    data = np.zeros((neq, 7))
    for i in range(neq):
        b1, b2 = E["b1"][i], E["b2"][i]
        R1 = q_to_mat(kin["xquat"][b1])
        data[i, :3] = R1.T @ (kin["xpos"][b2] - kin["xpos"][b1])
        data[i, 3:] = q_mul(q_conj(kin["xquat"][b1]), kin["xquat"][b2])
    m.a["eq_data"] = data
    m.a["collision_pairs"] = _collision_pairs(m)
    return m


# --------------------------------------------------------------------------------------
# compile-time constants that need kinematics / inertia at qpos0 (the mj_setConst step)
# --------------------------------------------------------------------------------------


def kinematics_np(m, qpos):
    """Plain numpy forward kinematics; compile-time use only (invweight0, weld relpose, tests)."""
    nb = m.nbody
    xpos = np.zeros((nb, 3))
    xquat = np.zeros((nb, 4))
    xquat[0, 0] = 1
    xanchor = np.zeros((m.njnt, 3))
    xaxis = np.zeros((m.njnt, 3))
    for b in range(1, nb):
        p = m.body_parentid[b]
        ja, jn = m.body_jntadr[b], m.body_jntnum[b]
        if jn == 1 and m.jnt_type[ja] == JNT_FREE:
            qa = m.jnt_qposadr[ja]
            xpos[b] = qpos[qa : qa + 3]
            xquat[b] = q_norm(qpos[qa + 3 : qa + 7])
            xanchor[ja] = xpos[b]
            xaxis[ja] = q_to_mat(xquat[b])[:, 2]
            continue
        Rp = q_to_mat(xquat[p])
        pos = xpos[p] + Rp @ m.body_pos[b]
        quat = q_mul(xquat[p], m.body_quat[b])
        for j in range(ja, ja + jn):
            R = q_to_mat(quat)
            xanchor[j] = pos + R @ m.jnt_pos[j]
            xaxis[j] = R @ m.jnt_axis[j]
            q = qpos[m.jnt_qposadr[j]] - m.qpos0[m.jnt_qposadr[j]]
            if m.jnt_type[j] == JNT_HINGE:
                quat = q_mul(quat, q_axis_angle(m.jnt_axis[j], q))
                pos = xanchor[j] - q_to_mat(quat) @ m.jnt_pos[j]
            else:
                pos = pos + xaxis[j] * q
        xpos[b] = pos
        xquat[b] = q_norm(quat)
    xmat = np.array([q_to_mat(q) for q in xquat])
    xipos = np.array([xpos[b] + xmat[b] @ m.body_ipos[b] for b in range(nb)])
    ximat = np.array([q_to_mat(q_mul(xquat[b], m.body_iquat[b])) for b in range(nb)])
    return dict(xpos=xpos, xquat=xquat, xmat=xmat, xipos=xipos, ximat=ximat, xanchor=xanchor, xaxis=xaxis)


def _dof_jacobian_np(m, kin, body, point):
    """6 x nv Jacobian (rows 0-2 translational at `point`, rows 3-5 rotational) of `body`."""
    Jm = np.zeros((6, m.nv))
    b = body
    while b > 0:
        for j in range(m.body_jntadr[b], m.body_jntadr[b] + m.body_jntnum[b]):
            da = m.jnt_dofadr[j]
            t = m.jnt_type[j]
            if t == JNT_FREE:
                Jm[0:3, da : da + 3] = np.eye(3)
                R = kin["xmat"][b]
                for k in range(3):
                    ax = R[:, k]
                    Jm[3:6, da + 3 + k] = ax
                    Jm[0:3, da + 3 + k] = np.cross(ax, point - kin["xpos"][b])
            elif t == JNT_HINGE:
                ax = kin["xaxis"][j]
                Jm[3:6, da] = ax
                Jm[0:3, da] = np.cross(ax, point - kin["xanchor"][j])
            else:
                Jm[0:3, da] = kin["xaxis"][j]
        b = m.body_parentid[b]
    return Jm


def mass_matrix_np(m, kin):
    """Dense joint-space inertia via sum_b J_b^T I_b J_b (slow, compile-time only)."""
    M = np.zeros((m.nv, m.nv))
    for b in range(1, m.nbody):
        if m.body_mass[b] == 0 and not np.any(m.body_inertia[b]):
            continue
        Jb = _dof_jacobian_np(m, kin, b, kin["xipos"][b])
        Rw = kin["ximat"][b]
        Iw = Rw @ np.diag(m.body_inertia[b]) @ Rw.T
        M += m.body_mass[b] * Jb[:3].T @ Jb[:3] + Jb[3:].T @ Iw @ Jb[3:]
    M += np.diag(m.dof_armature)
    return M


def _set_const(m):
    """body_invweight0 / dof_invweight0 / stat_meaninertia at qpos0 (MuJoCo's mj_setConst semantics:
    invweight0[b] = mean diagonal of J M^-1 J^T for the translational / rotational body Jacobian at the
    body CoM; dof_invweight0 = diag(M^-1), averaged over the 3+3 dofs of a free joint)."""
    kin = kinematics_np(m, m.qpos0)
    nv = m.nv
    M = mass_matrix_np(m, kin)
    m.a["stat_meaninertia"] = float(np.mean(np.diag(M))) if nv else 1.0
    Minv = np.linalg.inv(M) if nv else np.zeros((0, 0))
    bw = np.zeros((m.nbody, 2))
    for b in range(1, m.nbody):
        if m.body_weldid[b] == 0:
            continue
        Jb = _dof_jacobian_np(m, kin, b, kin["xipos"][b])
        A = Jb @ Minv @ Jb.T
        bw[b, 0] = max(MJ_MINVAL, np.trace(A[:3, :3]) / 3)
        bw[b, 1] = max(MJ_MINVAL, np.trace(A[3:, 3:]) / 3)
    m.a["body_invweight0"] = bw
    dw = np.diag(Minv).copy() if nv else np.zeros(0)
    for j in range(m.njnt):
        if m.jnt_type[j] == JNT_FREE:
            da = m.jnt_dofadr[j]
            dw[da : da + 3] = np.mean(dw[da : da + 3])
            dw[da + 3 : da + 6] = np.mean(dw[da + 3 : da + 6])
    m.a["dof_invweight0"] = dw


def _collision_pairs(m):
    """Static part of MuJoCo's pair filtering, resolved at compile time: same body, welded-together
    bodies, parent-child (world exempt), both welded to world, <exclude>, and geoms that can never
    collide (contype=conaffinity=0 is NOT filtered here: masks are per-env run-time state)."""
    pairs = []
    excl = set((int(a), int(b)) for a, b in m.exclude) | set((int(b), int(a)) for a, b in m.exclude)
    for g1 in range(m.ngeom):
        for g2 in range(g1 + 1, m.ngeom):
            b1, b2 = int(m.geom_bodyid[g1]), int(m.geom_bodyid[g2])
            w1, w2 = int(m.body_weldid[b1]), int(m.body_weldid[b2])
            if b1 == b2 or w1 == w2:
                continue
            wp1 = int(m.body_weldid[m.body_parentid[w1]])
            wp2 = int(m.body_weldid[m.body_parentid[w2]])
            if w1 != 0 and w2 != 0 and (w1 == wp2 or w2 == wp1):
                continue
            if (b1, b2) in excl:
                continue
            if m.geom_type[g1] == GEOM_PLANE and m.geom_type[g2] == GEOM_PLANE:
                continue
            pairs.append((g1, g2))
    return np.array(pairs, dtype=np.int32).reshape(len(pairs), 2)


def load_recipe(furniture, assets_root):
    """the assembly recipe of a furniture model (FurnitureEnv._load_recipe, furniture.py:2033-2044): assets/recipes/<name>.yaml with
    python/tuple tags read as lists; None when the model has no recipe.  Kept in the compiled scene as JSON (meta["recipe_json"])."""
    path = os.path.join(assets_root, "recipes", furniture + ".yaml")
    if not os.path.exists(path):
        return None
    import yaml

    class _Loader(yaml.SafeLoader):
        pass

    _Loader.add_constructor("tag:yaml.org,2002:python/tuple", lambda loader, node: loader.construct_sequence(node))
    with open(path) as f:
        return yaml.load(f, Loader=_Loader)


def compose_agent(agent, furniture, assets_root, resize_factor=None):
    """compose_scene with the agent names of the compiled tables: "SawyerTorque" is the Sawyer on torque (motor) actuators,
    robots/sawyer/robot_torque.xml -- what the reference loads for control_type "torque" and the NEW_CONTROLLERS (furniture.py:1893-1899)"""
    if agent == "SawyerTorque":
        xml, meta = compose_scene("Sawyer", furniture, assets_root, resize_factor=resize_factor, use_torque=True)
        meta["agent"] = "SawyerTorque"
        return xml, meta
    return compose_scene(agent, furniture, assets_root, resize_factor=resize_factor)


def load_scene(agent="Sawyer", furniture="table_lack_0825", assets_root=None, resize_factor=None):
    """compose + compile if the asset tree is reachable, else the precompiled tables shipped in
    furniture_b200/compiled/ (made by tools/compile_models.py; unit size only)."""
    root = assets_root or default_assets_root()
    if root is not None:
        xml, meta = compose_agent(agent, furniture, root, resize_factor=resize_factor)
        return compile_mjcf(xml, meta)
    if resize_factor:
        raise FileNotFoundError("a resized scene (furn_size_rand) is composed from the MJCF asset tree: set FURNITURE_ASSETS")
    path = os.path.join(os.path.dirname(__file__), "compiled", "%s_%s.npz" % (agent, furniture))
    if not os.path.exists(path):
        raise FileNotFoundError("no asset tree and no compiled model at " + path)
    return Model.load(path)
