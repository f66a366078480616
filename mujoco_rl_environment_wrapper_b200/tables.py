"""Index tables derived once from the MJCF + config with the reference's own rules.

Restates (does not import) the table builders of the reference:
  observation indices   MuJoCo_Gym/mujoco_parent.py:233-272, :185-231, :139-183; sensor.py:1-116
  action indices        MuJoCo_Gym/mujoco_parent.py:274-314
  action routing        MuJoCo_Gym/mujoco_rl.py:171-193
The reference walks an xmltodict tree; here the same traversal order (document order, depth first)
is taken over ElementTree.
"""
import xml.etree.ElementTree as ET

from . import _lib as L

SENSOR_DIM = {"touch": 1, "accelerometer": 3, "rangefinder": 1, "framexaxis": 3, "frameyaxis": 3, "framezaxis": 3,
              "velocimeter": 3, "gyro": 3, "jointpos": 1, "jointvel": 1, "framepos": 3, "framequat": 4, "framelinvel": 3,
              "frameangvel": 3}
# the attribute naming a sensor's object ("objname" with "objtype" for the frame sensors)
_SITE_SENSORS = ("touch", "accelerometer", "rangefinder", "velocimeter", "gyro")
_JOINT_SENSORS = ("jointpos", "jointvel")


def _iter_bodies(elem):
    for b in elem.findall("body"):
        yield b
        yield from _iter_bodies(b)


def find_body(root, name):
    wb = root.find("worldbody")
    for b in _iter_bodies(wb):
        if b.get("name") == name:
            return b
    raise Exception(f"Agent body '{name}' not found in the MJCF")


def _subtree_elems(body, tag):
    out = list(body.findall(tag))
    for b in body.findall("body"):
        out += _subtree_elems(b, tag)
    return out


def sensor_space(kind, cutoff):
    """(low, high) lists for one sensor, sensor.py:64-116."""
    if kind == "touch":
        return [0], [float(cutoff)]
    if kind == "accelerometer" and cutoff is not None:
        return [-float(cutoff)] * 3, [float(cutoff)] * 3
    if kind == "rangefinder":
        return [-1], [float(cutoff)]
    if kind in ("framexaxis", "frameyaxis", "framezaxis"):
        return [-1] * 3, [1] * 3
    if kind == "framequat":
        return [-1] * 4, [1] * 4
    if kind in SENSOR_DIM:   # real-valued: clamped to +-cutoff when cutoff > 0
        c = float(cutoff) if cutoff is not None else 0.0
        b = c if c > 0 else float("inf")
        return [-b] * SENSOR_DIM[kind], [b] * SENSOR_DIM[kind]
    raise Exception(f"unsupported sensor type {kind}")


class Tables:
    def __init__(self, xml_text, model: "L.Model", agents, free_joint):
        self.root = ET.fromstring(xml_text)
        self.model = model
        wb = self.root.find("worldbody")
        # every NAMED joint under <worldbody>, document order == joint id order (mujoco_parent.py:246-257)
        f = model.fields
        qpos_idx, qvel_idx = [], []
        joints = []

        def walk(body):
            for j in body.findall("joint"):
                joints.append(j)
            for fj in body.findall("freejoint"):
                joints.append(fj)
            for b in body.findall("body"):
                walk(b)
        walk(wb)
        for j in joints:
            name = j.get("name")
            if not name:
                continue
            jid = model.name2id(L.OBJ_JOINT, name)
            if jid < 0:
                raise Exception(f"joint {name} not found in the compiled model")
            qa, da = int(f["jnt_qposadr"][jid]), int(f["jnt_dofadr"][jid])
            free = int(f["jnt_type"][jid]) == L.JNT_FREE
            qpos_idx += list(range(qa, qa + (7 if free else 1)))
            qvel_idx += list(range(da, da + (6 if free else 1)))
        self.qpos_idx, self.qvel_idx = qpos_idx, qvel_idx
        # sensors in sensor-id order with their sensordata addresses (sensor.py:42-61)
        self.sensors = []
        sens = self.root.find("sensor")
        if sens is not None:
            adr = 0
            for s in list(sens):
                kind = s.tag
                if kind not in SENSOR_DIM:
                    raise Exception(f"unsupported sensor <{kind}>")
                if kind in _SITE_SENSORS:
                    objtype, obj = "site", s.get("site")
                elif kind in _JOINT_SENSORS:
                    objtype, obj = "joint", s.get("joint")
                else:
                    objtype, obj = s.get("objtype"), s.get("objname")
                self.sensors.append({"name": s.get("name"), "type": kind, "objtype": objtype, "obj": obj, "cutoff": s.get("cutoff"),
                                     "indices": list(range(adr, adr + SENSOR_DIM[kind]))})
                adr += SENSOR_DIM[kind]
        self.agents_observation_index, self.agents_action_index = {}, {}
        self.obs_space, self.act_space, self.agent_body = {}, {}, {}
        self.rgb_sensors = {}   # agent -> names of the cameras in its subtree (mujoco_parent.py:505-516)
        motors = []
        act = self.root.find("actuator")
        if act is not None:
            motors = list(act.findall("motor"))
        for agent in agents:
            body = find_body(self.root, agent)
            self.agent_body[agent] = model.name2id(L.OBJ_BODY, agent)
            self.rgb_sensors[agent] = [c.get("name") for c in _subtree_elems(body, "camera")]
            # a sensor belongs to the agent whose subtree holds its object
            owned = {t: {e.get("name") for e in _subtree_elems(body, t)} for t in ("site", "joint", "geom")}
            owned["body"] = owned["xbody"] = {body.get("name")} | {e.get("name") for e in _subtree_elems(body, "body")}
            mine = [s for s in self.sensors if s["obj"] in owned.get(s["objtype"], ())]
            s_idx = [i for s in mine for i in s["indices"]]
            low, high = [], []
            for s in mine:
                lo, hi = sensor_space(s["type"], s["cutoff"])
                low += lo
                high += hi
            inf = float("inf")
            low += [-inf] * (len(qpos_idx) + len(qvel_idx))
            high += [inf] * (len(qpos_idx) + len(qvel_idx))
            self.agents_observation_index[agent] = {"sensors": s_idx, "qpos": list(qpos_idx), "qvel": list(qvel_idx)}
            self.obs_space[agent] = {"low": low, "high": high}
            # actions (mujoco_parent.py:274-314)
            if free_joint:
                own = body.findall("joint") + body.findall("freejoint")
                if not own:
                    raise Exception(f"The agent {agent} has to have a free joint")
                fj = own[0]
                if (fj.tag != "freejoint") and fj.get("type") != "free":
                    raise Exception(f"The joint of agent {agent} has to be of type free")
                jid = model.name2id(L.OBJ_JOINT, fj.get("name"))
                d = int(f["jnt_dofadr"][jid])
                self.agents_action_index[agent] = [d, d + 1, d + 5]
                self.act_space[agent] = {"low": [-1, -1, -1], "high": [1, 1, 1]}
            else:
                idx, lo, hi = [], [], []
                for j in _subtree_elems(body, "joint"):
                    for k, mtr in enumerate(motors):
                        if mtr.get("joint") == j.get("name"):
                            idx.append(k)
                            cr = (mtr.get("ctrlrange") or "0 0").split()
                            lo.append(float(cr[0]))
                            hi.append(float(cr[1]))
                self.agents_action_index[agent] = idx
                self.act_space[agent] = {"low": lo, "high": hi}
