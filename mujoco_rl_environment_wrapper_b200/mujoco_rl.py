"""Drop-in `MuJoCoRL` over the batched CUDA step path.

Mirrors the reference's public surface (MuJoCo_Gym/mujoco_rl.py:18-430, mujoco_parent.py:19-478):
`MuJoCoRL(config_dict)`, `reset()`, `step(action_dict)`, `action_space(agent)`,
`observation_space(agent)`, `filter_by_tag`, `get_data`, `distance`, `collision`,
`get_observations`, `get_sensor_data`, attributes `agents`, `possible_agents`, `data_store`,
`timestep`, `max_steps`, `skip_frames`, `action_routing`, `agents_action_index`,
`agents_observation_index`.

New optional config keys: `num_envs` (default 1), `device`, `seed`, `autoReset` (default False: `step()` resets every
env whose episode it ends, in the same kernel launch; see `step`), `startStates` ({"qpos": [P, nq], "qvel": [P, nv]}:
every reset starts from a pool row drawn per env and reset instead of qpos0; see `reset`), `perEnvParams` (True: every
env has its own body masses / inertias, geom frictions, actuator gears and dof dampings, `env.params`) and
`randomizeParams` ({"body_mass": [lo, hi], "geom_friction": ..., "actuator_gear": ..., "dof_damping": ...}: every reset
scales the env's parameters by factors drawn in [lo, hi]; implies `perEnvParams`).  Positions of the agents' bodies and of
the `filter_by_tag("target")` objects are exported every step (`distance`, `get_data`).  With `num_envs == 1` results are squeezed to the
reference's shapes (numpy arrays, Python scalars); otherwise every per-agent value is a CUDA tensor
with a leading `num_envs` dimension.  There is no CPU path: construction raises without a GPU.
"""
import ctypes
import json
import os
import random

import numpy as np
import torch

from . import _lib as L
from .batch import Batch
from .dataview import DataView, ModelView, quat_to_euler_zyx_deg, static_pose
from .plugins import recognise
from .spaces import Box
from .tables import Tables


class AgentStore(dict):
    """`env.data_store[agent]`: plain dict for user plugins; the fused plugins' keys are views of the
    device store columns (`utterance`, `current_target`, `inventory`, `distance`, `xpos_before`)."""

    def __init__(self, env, a):
        super().__init__()
        self._env, self._a = env, a

    def _col(self, key):
        b = self._env._batch
        if key in ("utterance", "inventory"):
            return b.store_i[:, self._a, L.STORE_I[key]]
        if key == "current_target":
            return b.store_i[:, self._a, L.STORE_I["current_target"]] - 1
        if key in L.STORE_F:
            return b.store_f[:, self._a, L.STORE_F[key]]
        return None

    def __missing__(self, key):
        col = self._col(key)
        if col is None:
            raise KeyError(key)
        return col if self._env.num_envs > 1 else col[0].item()


def state_rows(what, v, rows, width, device):
    """float32 tensor [rows, width] on `device` from a numpy array or tensor; rows = None: any count >= 1; with rows = 1
    a single row [width] is accepted too"""
    t = (v if torch.is_tensor(v) else torch.as_tensor(np.asarray(v, dtype=np.float32))).to(device, torch.float32)
    if rows == 1 and t.dim() == 1:
        t = t.reshape(1, -1)
    if t.dim() != 2 or t.shape[1] != width or (rows is None and t.shape[0] < 1) or (rows is not None and t.shape[0] != rows):
        want = f"[{'P >= 1' if rows is None else rows}, {width}]" + (f" (or [{width}])" if rows == 1 else "")
        raise Exception(f"{what}: expected shape {want}, got {tuple(t.shape)}")
    return t.contiguous()


def parse_param_ranges(cfg):
    """config "randomizeParams" {family: [lo, hi]} -> four (lo, hi) in L.PARAM_FAMILIES order (missing: (1, 1)), or None"""
    if cfg is None:
        return None
    if not isinstance(cfg, dict) or any(k not in L.PARAM_FAMILIES for k in cfg):
        raise Exception(f"randomizeParams: expected a dict with keys among {list(L.PARAM_FAMILIES)}, got {cfg!r}")
    out = []
    for f in L.PARAM_FAMILIES:
        r = cfg.get(f, (1.0, 1.0))
        try:
            lo, hi = (float(x) for x in r)
        except (TypeError, ValueError):
            raise Exception(f"randomizeParams['{f}']: expected [lo, hi], got {r!r}")
        if not (np.isfinite(lo) and np.isfinite(hi)) or lo > hi or lo < 0 or (f == "body_mass" and lo <= 0):
            raise Exception(f"randomizeParams['{f}']: need finite 0 {'<' if f == 'body_mass' else '<='} lo <= hi, got [{lo}, {hi}]")
        out.append((lo, hi))
    return out


def parse_start_states(cfg, nq, nv, device):
    """config "startStates" {"qpos": [P, nq], "qvel": [P, nv] (optional, zeros)} -> (qpos, qvel) tensors, or None"""
    if cfg is None:
        return None
    if not isinstance(cfg, dict) or cfg.get("qpos") is None:
        raise Exception('startStates: expected {"qpos": [P, nq], "qvel": [P, nv] (optional)}')
    qpos = state_rows("startStates['qpos']", cfg["qpos"], None, nq, device)
    qvel = state_rows("startStates['qvel']", cfg["qvel"], qpos.shape[0], nv, device) if cfg.get("qvel") is not None \
        else torch.zeros((qpos.shape[0], nv), dtype=torch.float32, device=device)
    if not bool(torch.isfinite(qpos).all() and torch.isfinite(qvel).all()):
        raise Exception("startStates: qpos / qvel must be finite")
    return qpos, qvel


class MuJoCoRL:
    metadata = {"name": "mujoco_rl_b200"}

    def __init__(self, config_dict: dict):
        self.agents = config_dict.get("agents", [])
        self.possible_agents = self.agents
        self.xml_paths = config_dict.get("xmlPath")
        self.info_jsons = config_dict.get("infoJson", None)
        self.render_mode = config_dict.get("renderMode", False)
        self.export_path = config_dict.get("exportPath")
        self.free_joint = config_dict.get("freeJoint", False)
        self.skip_frames = config_dict.get("skipFrames", 1)
        self.max_steps = config_dict.get("maxSteps", 1024)
        self.reward_functions = list(config_dict.get("rewardFunctions", []))
        self.done_functions = list(config_dict.get("doneFunctions", []))
        dynamics_classes = list(config_dict.get("environmentDynamics", []))
        self.agent_cameras = config_dict.get("agentCameras", False)
        self.sensor_resolution = tuple(config_dict.get("sensorResolution", (64, 64)))
        self.num_envs = int(config_dict.get("num_envs", 1))
        self.seed = int(config_dict.get("seed", 1234))
        self.reset_noise = float(config_dict.get("resetNoise", 0.0))   # new, off: the reference restarts at qpos0
        self.auto_reset = bool(config_dict.get("autoReset", False))     # new, off: the reference's loop resets by hand
        # new: names of further bodies / geoms whose positions (and orientations) are exported every step, or "all";
        # agents, "target"-tagged objects and static objects are always available to distance / get_data / data.body(n)
        self.export_positions = config_dict.get("exportPositions", [])
        # orientations of the exported moving objects (get_data()["orientation"]); default: on for the drop-in
        # single env, off for batches (16 bytes per object and env-step)
        self.export_orientation = bool(config_dict.get("exportOrientation", self.num_envs == 1 or bool(self.export_positions)))
        dev = config_dict.get("device", None)
        if not torch.cuda.is_available():
            raise RuntimeError("MuJoCoRL (B200): no CUDA device available; this implementation has no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if dev is None else torch.device(dev)
        if not self.agents:
            raise Exception("config_dict['agents'] must name at least one agent body")
        if len(self.agents) > L.MAX_AGENTS:
            raise Exception(f"at most {L.MAX_AGENTS} agents are supported")

        self.timestep = 0
        self.action_routing = {"physical": [], "dynamic": {}}
        # xml: str, or list = level variants re-drawn at every reset (mujoco_parent.py:88-91, 351-356).  Every level
        # is compiled once; with num_envs > 1 each env carries its own level id.
        self._level_paths = [self.xml_paths] if isinstance(self.xml_paths, str) else list(self.xml_paths)
        if isinstance(self.info_jsons, list) and len(self.info_jsons) != len(self._level_paths):
            raise Exception("Length mismatch between info_json list and xml_paths list")
        self._level_rng = np.random.default_rng(self.seed)
        self._levels = []
        for path in self._level_paths:
            with open(path, "r") as fh:
                text = fh.read()
            model = ModelView(L.Model(text))
            tables = Tables(text, model, self.agents, self.free_joint)
            info_json, names = self.__load_json(path)
            self._levels.append({"xml_path": path, "xml_text": text, "model": model, "tables": tables,
                                 "info_json": info_json, "info_name_list": names})
        first = self._levels[0]["tables"]
        for lv in self._levels[1:]:
            t, m, m0 = lv["tables"], lv["model"], self._levels[0]["model"]
            if (t.agents_action_index != first.agents_action_index or t.agents_observation_index != first.agents_observation_index
                    or t.obs_space != first.obs_space or t.act_space != first.act_space
                    or (m.nq, m.nv, m.nu, m.nsensordata) != (m0.nq, m0.nv, m0.nu, m0.nsensordata)):
                raise Exception(f"level '{lv['xml_path']}' is not structurally identical to '{self._levels[0]['xml_path']}' "
                                f"(the reference builds its index tables once and reuses them for every level)")
        self._first_level = self._level_paths.index(random.choice(self._level_paths)) if self.num_envs == 1 else 0
        self._use_level(self._first_level)
        self._start_states = parse_start_states(config_dict.get("startStates"), self.model.nq, self.model.nv, self.device)
        self._param_ranges = parse_param_ranges(config_dict.get("randomizeParams"))
        self._per_env_params = bool(config_dict.get("perEnvParams", False)) or self._param_ranges is not None
        if self._per_env_params and int(self.skip_frames) == 0:
            raise Exception("perEnvParams / randomizeParams need skipFrames >= 1 (the physics-free step reads no parameter)")
        self.agents_action_index = self._tables.agents_action_index
        self.agents_observation_index = self._tables.agents_observation_index

        self.data_store = {agent: AgentStore(self, a) for a, agent in enumerate(self.agents)}
        self.data = DataView(self)
        self.environment_dynamics = [dyn(self) for dyn in dynamics_classes]
        self.__build_spaces()
        self.__build_batch()
        # the reference validates every plugin by calling it once (mujoco_rl.py:114-169); whatever that call writes is
        # discarded again (store, draw counters), so that construction does not consume random draws
        b = self._batch
        snap = (b.store_i.clone(), b.store_f.clone())
        # (plugins fused through their verbatim reference source are not called: their code is written for one env)
        own = lambda obj: hasattr(obj, "mjb_kind")
        self.__check_dynamics([d for d in self.environment_dynamics if d not in self._fused_dyn or own(d.__class__)])
        self.__check_reward_functions([fn for fn in self.reward_functions if fn in self._host_rew or own(fn)])
        self.__check_done_functions([fn for fn in self.done_functions if fn in self._host_done or own(fn)])
        b.store_i.copy_(snap[0]); b.store_f.copy_(snap[1])
        self._wipe_store()

    # ------------------------------------------------------------------------------------------
    def __load_json(self, xml_path):
        """mujoco_rl.py:93-112: the info JSON that belongs to `xml_path` (list entries are matched by file stem)"""
        src = self.info_jsons
        if isinstance(src, list):
            stem = os.path.split(xml_path)[1].split(".")[0] + ".json"
            src = [cur for cur in src if stem in cur][0]
        if isinstance(src, str):
            with open(src) as fh:
                info = json.load(fh)
        elif isinstance(src, dict):  # convenience: already-parsed json
            info = src
        else:
            return None, []
        return info, list(info["environment"]["objects"].keys())

    def _use_level(self, lid):
        """the attributes the reference re-binds when it (re)loads a level (mujoco_parent.py:351-356, mujoco_rl.py:304-310)"""
        lv = self._levels[lid]
        self.xml_path, self._xml_text, self.model, self._tables = lv["xml_path"], lv["xml_text"], lv["model"], lv["tables"]
        self.info_json, self.info_name_list = lv["info_json"], lv["info_name_list"]
        if "probe_names" in lv:
            self._target_names, self._probe_names = lv["target_names"], lv["probe_names"]

    def __build_spaces(self):
        """mujoco_rl.py:171-213"""
        self._observation_space, self._action_space = {}, {}
        self._n_mj_obs = {}
        for agent in self.agents:
            osp = {k: list(v) for k, v in self._tables.obs_space[agent].items()}
            self._n_mj_obs[agent] = len(osp["low"])
            asp = {k: list(v) for k, v in self._tables.act_space[agent].items()}
            self.action_routing["physical"] = [0, len(asp["low"])]
            for dyn in self.environment_dynamics:
                n0 = len(asp["low"])
                self.action_routing["dynamic"][dyn.__class__.__name__] = [n0, n0 + len(dyn.action_space["low"])]
                asp["low"] += list(dyn.action_space["low"])
                asp["high"] += list(dyn.action_space["high"])
                osp["low"] += list(dyn.observation_space["low"])
                osp["high"] += list(dyn.observation_space["high"])
            self._observation_space[agent] = Box(low=np.array(osp["low"], dtype=np.float32), high=np.array(osp["high"], dtype=np.float32))
            self._action_space[agent] = Box(low=np.array(asp["low"], dtype=np.float32), high=np.array(asp["high"], dtype=np.float32))
        n_phys = {len(self._tables.act_space[a]["low"]) for a in self.agents}
        if len(n_phys) != 1:
            raise Exception("all agents must have the same number of physical actions (mujoco_rl.py:182)")

    def _targets(self):
        if self.info_json is None:
            return []
        try:
            return self.__filter_names("target")
        except KeyError:
            return []

    def __filter_names(self, tag):
        """names in filter_by_tag order, duplicates kept (mujoco_rl.py:355-378)"""
        names = []
        objs = self.info_json["environment"]["objects"]
        for obj in objs:
            if "tags" in objs[obj].keys() and objs[obj]["tags"] is not None and tag in objs[obj]["tags"]:
                names.append(obj)
        for area in self.info_json["areas"]:
            aobjs = self.info_json["areas"][area]["objects"]
            for obj in aobjs:
                if "tags" in aobjs[obj].keys() and aobjs[obj]["tags"] is not None and tag in aobjs[obj]["tags"]:
                    names.append(obj)
        return names

    def _resolve(self, name):
        """name -> (objtype, id) with the reference's body-then-geom fallback (mujoco_parent.py:403-425)"""
        bid = self.model.name2id(L.OBJ_BODY, name)
        if bid >= 0:
            return L.OBJ_BODY, bid
        gid = self.model.name2id(L.OBJ_GEOM, name)
        if gid >= 0:
            return L.OBJ_GEOM, gid
        raise KeyError(f"Invalid name '{name}': neither a body nor a geom")

    def __build_batch(self):
        """one spec + batch handle per level over ONE set of tensors; single-level envs keep env packing"""
        multi = len(self._levels) > 1
        if self.auto_reset and multi:
            raise Exception("autoReset: an xmlPath list with several levels is not supported (a reset draws the env's level "
                            "on the host)")
        if self.auto_reset and int(self.skip_frames) == 0:
            raise Exception("autoReset needs skipFrames >= 1 (the physics-free step has no forward pass to reset with)")
        for lid, lv in enumerate(self._levels):
            self._use_level(lid)
            spec, keep = self.__build_spec()
            if multi:
                spec.flags |= L.SPEC_NO_PACK
            if self.auto_reset:
                host = [getattr(p, "__name__", p.__class__.__name__) for p in
                        [d for d, _, _ in self._host_dyn] + self._host_rew + self._host_done]
                if host:
                    raise Exception(f"autoReset: plugins that run as host code after the kernel are not supported ({host}): "
                                    f"they would read the new episode's state of an env the step reset")
                spec.flags |= L.SPEC_AUTORESET
                asp = self._action_space[self.agents[0]]   # homogeneous across agents, as sample_actions assumes
                for d in range(self._act_dim):
                    spec.act_low[d], spec.act_high[d] = float(asp.low[d]), float(asp.high[d])
            lv["spec"], lv["target_names"], lv["probe_names"] = spec, self._target_names, self._probe_names
            with torch.cuda.device(self.device):
                lv["batch"] = Batch(self.model, spec, self.num_envs, device=self.device, keepalive=keep,
                                    share=self._levels[0]["batch"] if lid else None, probe_quat=self.export_orientation,
                                    start_states=self._start_states, params=self._per_env_params, param_ranges=self._param_ranges,
                                    final_qpos=self.auto_reset and bool(self.agent_cameras))
        self._use_level(0)
        self._spec, self._batch = self._levels[0]["spec"], self._levels[0]["batch"]
        self.params = self.__param_views() if self._per_env_params else None
        self.level_id = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)
        self._level_host = np.zeros(self.num_envs, dtype=np.int64)
        if multi:
            self._draw_levels(None, first=True)
        self._sample_gen = torch.Generator(device=self.device)
        self._sample_gen.manual_seed(self.seed)
        self._act_low = torch.tensor(np.asarray(self._action_space[self.agents[0]].low), device=self.device)
        self._act_high = torch.tensor(np.asarray(self._action_space[self.agents[0]].high), device=self.device)

    def __param_views(self):
        """`env.params`: writable views of the per-env parameter table (include/mjb.h, mjb_env_spec.params), MuJoCo id
        order: body_mass [N, nbody], body_inertia [N, nbody, 3], geom_friction [N, ngeom], actuator_gear [N, nu],
        dof_damping [N, nv]; the leading dimension is dropped for num_envs == 1.  Writes take effect at the next launch;
        with randomizeParams every reset overwrites the rows of the envs it resets.  With an `xmlPath` list the levels share
        the table; an env that moves to another level gets that level's values.  `env.model` keeps the nominal values."""
        t, off, m = self._batch.params, self._batch.param_offsets, self.model
        n = {"body_mass": m.nbody, "body_inertia": 3 * m.nbody, "geom_friction": m.ngeom, "actuator_gear": m.nu, "dof_damping": m.nv}
        views = {}
        for f in L.PARAM_FIELDS:
            v = t[:, off[f]:off[f] + n[f]]
            if f == "body_inertia":
                v = v.unflatten(1, (m.nbody, 3))
            views[f] = v if self.num_envs > 1 else v[0]
        return views

    def _draw_levels(self, mask, first=False):
        """a fresh level for every env being reset (the reference's random.choice at reset, mujoco_parent.py:351-352),
        then each level's handle is pointed at the envs it owns.  Host-side: resets are rare next to steps."""
        n_lv = len(self._levels)
        if self.num_envs == 1:   # one env: the reference's own draw (global `random`), already made once by __init__
            draw = np.array([self._first_level if first else self._level_paths.index(random.choice(self._level_paths))])
        else:
            draw = self._level_rng.integers(0, n_lv, size=self.num_envs)
        old = self._level_host
        if mask is None:
            self._level_host = draw
        else:
            m = mask.detach().to("cpu").numpy().astype(bool).reshape(-1)
            self._level_host = np.where(m, draw, self._level_host)
        self.level_id.copy_(torch.from_numpy(self._level_host.astype(np.int32)))
        if self._per_env_params and self._param_ranges is None:
            # the levels share one table: an env that moves to another level starts from that level's own values
            # (a randomising reset draws them from the level's image anyway)
            moved = np.ones(self.num_envs, bool) if first else self._level_host != old
            table = self._levels[0]["batch"].params
            for lid, lv in enumerate(self._levels):
                ids = np.nonzero(moved & (self._level_host == lid))[0]
                if len(ids):
                    row = torch.from_numpy(lv["model"].nominal_params()).to(table.device)
                    table[torch.from_numpy(ids).to(table.device)] = row
        for lid, lv in enumerate(self._levels):
            lv["batch"].set_subset(torch.from_numpy(np.nonzero(self._level_host == lid)[0].astype(np.int32)))
        self._use_level(int(self._level_host[0]))

    def __build_spec(self):
        A = len(self.agents)
        spec = L.EnvSpec()
        spec.n_agents, spec.free_joint = A, int(bool(self.free_joint))
        spec.skip_frames, spec.max_steps = int(self.skip_frames), int(self.max_steps)
        n_phys = len(self._tables.act_space[self.agents[0]]["low"])
        spec.n_phys_act = n_phys
        act_index, obs_index, adr = [], [], [0]
        for a, agent in enumerate(self.agents):
            act_index += self.agents_action_index[agent]
            oi = self.agents_observation_index[agent]
            obs_index += [(0 << 24) | i for i in oi["sensors"]] + [(1 << 24) | i for i in oi["qpos"]] + [(2 << 24) | i for i in oi["qvel"]]
            adr.append(len(obs_index))
            spec.agent_body[a] = self._tables.agent_body[agent]
        for a in range(A + 1):
            spec.obs_adr[a] = adr[a]
        # plugins: fused kinds go to the kernel, the rest run as batched torch code after it
        self._fused_dyn, self._host_dyn, self._host_rew, self._host_done = [], [], [], []
        nd = nr = ndn = 0
        act_pos = n_phys
        fused_obs = 0
        # a plugin is fused when it is one of the reference's examples (marker or verbatim source, plugins.recognise)
        # and no host plugin precedes it in its list (the lists run in order)
        for dyn in self.environment_dynamics:
            kind = recognise(dyn.__class__)
            lo = act_pos
            act_pos += len(dyn.action_space["low"])
            if kind and kind[0] == "dynamic" and not self._host_dyn:
                p = spec.dynamics[nd]
                p.kind, p.act_lo, p.act_hi, p.n_obs = kind[1], lo, act_pos, len(dyn.observation_space["low"])
                p.param[0] = float(getattr(dyn, "threshold", kind[2].get("threshold", 0.0)))
                nd += 1
                fused_obs += p.n_obs
                self._fused_dyn.append(dyn)
            else:
                self._host_dyn.append((dyn, lo, act_pos))
        for fn in self.reward_functions:
            kind = recognise(fn)
            if kind and kind[0] == "reward" and not self._host_rew:
                p = spec.rewards[nr]
                p.kind = kind[1]
                p.param[0] = float(getattr(fn, "scale", kind[2].get("scale", 1.0)))
                nr += 1
            else:
                self._host_rew.append(fn)
        for fn in self.done_functions:
            kind = recognise(fn)
            if kind and kind[0] == "done" and not self._host_done:
                p = spec.dones[ndn]
                p.kind = kind[1]
                p.param[0] = float(getattr(fn, "threshold", kind[2].get("threshold", 1.0)))
                ndn += 1
            else:
                self._host_done.append(fn)
        spec.n_dynamics, spec.n_rewards, spec.n_dones = nd, nr, ndn
        spec.act_dim = act_pos
        self._act_dim = act_pos
        for a, agent in enumerate(self.agents):
            spec.obs_dim[a] = self._n_mj_obs[agent] + fused_obs
        self._fused_obs = fused_obs
        # targets (filter_by_tag("target")) and extra probes
        self._target_names = self._targets()
        if len(self._target_names) > L.MAX_TARGETS:
            raise Exception(f"at most {L.MAX_TARGETS} tagged targets are supported")
        self._probe_names = list(self.agents)
        spec.n_targets = len(self._target_names)
        for t, name in enumerate(self._target_names):
            ot, oid = self._resolve(name)
            spec.target_objtype[t], spec.target_objid[t] = ot, oid
            self._probe_names.append(name)
        extra = self.export_positions
        if extra == "all":
            m = self.model
            extra = [m.id2name(L.OBJ_BODY, i) for i in range(1, m.nbody)] + [m.id2name(L.OBJ_GEOM, i) for i in range(m.ngeom)]
            extra = [n for n in extra if n]
        n_x = 0
        for name in extra:
            if name in self._probe_names:
                continue
            ot, oid = self._resolve(name)
            if static_pose(self.model.fields, ot, oid) is not None:
                continue   # static: a constant, needs no slot
            if n_x >= L.MAX_EXTRA_PROBES:
                raise Exception(f"at most {L.MAX_EXTRA_PROBES} moving objects can be exported besides agents and targets")
            spec.extra_objtype[n_x], spec.extra_objid[n_x] = ot, oid
            self._probe_names.append(name)
            n_x += 1
        spec.n_extra_probes = n_x
        if any((recognise(fn) or (None, None))[:2] == ("reward", L.REW_ANT) for fn in self.reward_functions) and \
                any(int(t) == 1 for t in self.model.fields["sensor_type"]):
            raise Exception("ant_reward_function on a model with accelerometer sensors: MuJoCo then fills data.cfrc_ext and the "
                            "reward's contact-cost term is not zero; this term is not implemented")
        spec.seed = self.seed
        spec.reset_noise = float(self.reset_noise)
        self._ai = (ctypes.c_int32 * max(1, len(act_index)))(*act_index)
        self._oi = (ctypes.c_int32 * max(1, len(obs_index)))(*obs_index)
        spec.act_index = ctypes.cast(self._ai, ctypes.POINTER(ctypes.c_int32))
        spec.obs_index = ctypes.cast(self._oi, ctypes.POINTER(ctypes.c_int32))
        return spec, (self._ai, self._oi)

    # ---- validators (mujoco_rl.py:114-169): run each plugin once for agents[0]
    def __check_dynamics(self, dynamics):
        for dyn in dynamics:
            actions = dyn.action_space["low"]
            reward, observations, done, info = dyn.dynamic(self.agents[0], torch.tensor(actions, dtype=torch.float32, device=self.device).reshape(1, -1).expand(self.num_envs, -1))
            obs = torch.as_tensor(observations, dtype=torch.float32).reshape(-1, len(dyn.observation_space["low"])) if len(dyn.observation_space["low"]) else torch.zeros(1, 0)
            lo = torch.tensor(dyn.observation_space["low"], dtype=torch.float32, device=obs.device)
            hi = torch.tensor(dyn.observation_space["high"], dtype=torch.float32, device=obs.device)
            if obs.shape[-1] != len(dyn.observation_space["low"]):
                raise Exception(f"Observation, the second return variable of dynamic function, must match length"
                                f" of lower bound of observation space of {dyn}")
            if obs.numel() and not bool((obs >= lo).all()):
                raise Exception(f"Observation, the second return variable of dynamic function, exceeds the lower bound"
                                f" on at least one axis of the observation space of {dyn}")
            if obs.numel() and not bool((obs <= hi).all()):
                raise Exception(f"Observation, the second return variable of dynamic function, exceeds the upper bound"
                                f" on at least one axis of the observation space of {dyn}")
            if not (isinstance(reward, (int, float)) or torch.is_tensor(reward)):
                raise Exception(f"Reward, the first return variable of dynamic function of {dyn}, must be a float")

    def __check_done_functions(self, done_functions):
        for fn in done_functions:
            done = fn(self, self.agents[0])
            if not (isinstance(done, int) or torch.is_tensor(done)):
                raise Exception(f"Done, the first return variable of {fn}, must be a boolean")

    def __check_reward_functions(self, reward_functions):
        for fn in reward_functions:
            reward = fn(self, self.agents[0])
            if not (isinstance(reward, (int, float)) or torch.is_tensor(reward)):
                raise Exception(f"Reward, the second return variable of {fn}, must be a float")

    def _wipe_store(self, mask=None):
        """data_store = {agent: {}} (mujoco_rl.py:312,328) for all envs or the masked ones; the draw counters are not
        part of the store"""
        b = self._batch
        keep = b.store_i[:, :, L.STORE_I["draws"]].clone()
        if mask is None:
            b.store_i.zero_()
            b.store_f.zero_()
        else:
            m = mask.to(device=self.device, dtype=torch.bool).reshape(-1)
            b.store_i[m] = 0
            b.store_f[m] = 0
        b.store_i[:, :, L.STORE_I["draws"]] = keep
        for st in self.data_store.values():
            st.clear()

    # ------------------------------------------------------------------------------------------
    def action_space(self, agent):
        return self._action_space[agent]

    def observation_space(self, agent):
        return self._observation_space[agent]

    def sample_actions(self):
        """Uniform actions in [low, high) for every env and agent (device tensor [N, A, act_dim])."""
        u = torch.rand((self.num_envs, len(self.agents), self._act_dim), generator=self._sample_gen, device=self.device)
        return self._act_low + u * (self._act_high - self._act_low)

    def _load_actions(self, action):
        b = self._batch
        if torch.is_tensor(action):  # packed [N, A, act_dim]
            b.actions[:, :, :self._act_dim] = action.to(self.device, torch.float32).reshape(self.num_envs, len(self.agents), -1)
            return
        for a, agent in enumerate(self.agents):
            v = action[agent]
            t = v if torch.is_tensor(v) else torch.as_tensor(np.asarray(v, dtype=np.float32))
            b.actions[:, a, :self._act_dim] = t.to(self.device, torch.float32).reshape(-1, self._act_dim) if t.numel() else 0

    def _out(self, t):
        if self.num_envs > 1:
            return t
        return t[0].cpu().numpy().astype(np.float64) if t.dim() > 1 else t[0].item()

    def _collect_obs(self, extra):
        b = self._batch
        out = {}
        for a, agent in enumerate(self.agents):
            o = b.obs[:, a, :self._spec.obs_dim[a]]
            if extra and extra.get(agent):
                o = torch.cat([o] + extra[agent], dim=1)
            out[agent] = self._out(o)
        return out

    def step(self, action):
        """mujoco_rl.py:243-289 for all envs at once (one fused kernel launch).

        With `autoReset`, every env whose step ends with `term["__all__"] | trunc["__all__"]` is reset in the same launch,
        as `reset(mask=...)` would reset it, except that the dynamics see an action drawn in the kernel
        (include/mjb.h, mjb_reset_action) and reward / term / trunc stay those of the finishing step.  The returned
        observation of such an env is the new episode's first one; `infos[agent]["final_observation"]` holds the
        episode's last one (valid where `infos[agent]["_final_observation"]` is set).  Per-env step counters are
        `batch.timestep`; `self.timestep` counts calls."""
        b = self._batch
        self._load_actions(action)
        for lv in self._levels:
            lv["batch"].step()
        N = self.num_envs
        A = len(self.agents)
        flag = lambda t: t.view(torch.bool)   # the kernel writes 0 / 1 bytes: reinterpret, no extra kernel
        rewards = {agent: b.reward[:, a] for a, agent in enumerate(self.agents)}
        terms = {agent: flag(b.term[:, a]) for a, agent in enumerate(self.agents)}
        infos = {agent: {dyn.__class__.__name__: {} for dyn in self._fused_dyn} for agent in self.agents}
        extra = {agent: [] for agent in self.agents}
        for dyn, lo, hi in self._host_dyn:  # user dynamics as batched torch code, agent-inner order
            for a, agent in enumerate(self.agents):
                r, o, d, info = dyn.dynamic(agent, b.actions[:, a, lo:hi])
                extra[agent].append(torch.as_tensor(o, dtype=torch.float32, device=self.device).reshape(N, -1))
                rewards[agent] = rewards[agent] + r
                terms[agent] = terms[agent] | torch.as_tensor(d, device=self.device).bool()
                infos[agent][dyn.__class__.__name__] = info
        for fn in self._host_rew:
            rewards = {agent: rewards[agent] + fn(self, agent) for agent in self.agents}
        truncs = {agent: flag(b.trunc[:, a]) for a, agent in enumerate(self.agents)}
        truncs["__all__"] = flag(b.trunc[:, A])
        if self.done_functions:
            if self._host_done or self._host_dyn:
                for fn in self._host_done:
                    terms = {agent: terms[agent] | torch.as_tensor(fn(self, agent), device=self.device).bool() for agent in self.agents}
                allt = terms[self.agents[0]].clone()
                for agent in self.agents[1:]:
                    allt = allt | terms[agent]
                terms["__all__"] = allt
            else:
                terms["__all__"] = flag(b.term[:, A])   # the kernel's own OR over the agents
        self.timestep += 1
        obs = self._collect_obs(extra)
        if self.auto_reset:
            ended = (b.term[:, A] | b.trunc[:, A]).view(torch.bool)
            for a, agent in enumerate(self.agents):
                infos[agent]["final_observation"] = self._out(b.final_obs[:, a, :self._spec.obs_dim[a]])
                infos[agent]["_final_observation"] = ended if N > 1 else bool(ended[0].item())
        if N == 1:
            rewards = {k: (v[0].item() if torch.is_tensor(v) else v) for k, v in rewards.items()}
            if not self.environment_dynamics and not self.reward_functions:
                rewards = {k: 0 for k in rewards}   # the reference's untouched `int 0` (mujoco_rl.py:262)
            terms = {k: bool(v[0].item()) for k, v in terms.items()}
            truncs = {k: bool(v[0].item()) for k, v in truncs.items()}
        return obs, rewards, terms, truncs, infos

    def reset(self, *, seed=None, options=None, mask=None):
        """mujoco_rl.py:291-331.  `mask` (bool[N]) resets a subset of envs (new; the reference has one env).

        `options={"qpos": ..., "qvel": ...}` (new) starts the reset envs from these rows instead of qpos0 / zero velocity
        (or a `startStates` row): [N, nq] / [N, nv] for N > 1, [nq] / [nv] for N = 1; `qvel` defaults to zeros.  Rows of
        envs outside `mask` are ignored.  Everything else is an ordinary reset (include/mjb.h, mjb_reset_rows); rows are
        used as given (a free joint's quaternion comes back normalised, as after any forward pass)."""
        b = self._batch
        rows = options is not None and options.get("qpos") is not None
        if options is not None and not rows and options.get("qvel") is not None:
            raise Exception("reset(options=...): 'qvel' needs 'qpos'")
        if rows:
            N, nq, nv = self.num_envs, self.model.nq, self.model.nv
            qpos = state_rows("reset(options['qpos'])", options["qpos"], N, nq, self.device)
            qvel = state_rows("reset(options['qvel'])", options["qvel"], N, nv, self.device) if options.get("qvel") is not None \
                else torch.zeros((N, nv), dtype=torch.float32, device=self.device)
            if mask is None:
                b.qpos[:, :nq], b.qvel[:, :nv] = qpos, qvel
            else:
                m = mask.to(device=self.device, dtype=torch.bool).reshape(-1)
                b.qpos[m, :nq], b.qvel[m, :nv] = qpos[m], qvel[m]
        b.actions[:, :, :self._act_dim] = self.sample_actions()  # the reference applies dynamics once with a sampled action
        if len(self._levels) > 1:
            self._draw_levels(mask)
        for lv in self._levels:
            if rows:
                lv["batch"].reset_rows(mask)
            else:
                lv["batch"].reset(mask)
        for st in self.data_store.values():
            st.clear()
        infos = {agent: {dyn.__class__.__name__: {} for dyn in self._fused_dyn} for agent in self.agents}
        extra = {agent: [] for agent in self.agents}
        for dyn, lo, hi in self._host_dyn:
            for a, agent in enumerate(self.agents):
                r, o, d, info = dyn.dynamic(agent, b.actions[:, a, lo:hi])
                extra[agent].append(torch.as_tensor(o, dtype=torch.float32, device=self.device).reshape(self.num_envs, -1))
                infos[agent][dyn.__class__.__name__] = info
        if self._host_dyn:
            self._wipe_store(mask)   # everything the dynamics wrote is discarded (mujoco_rl.py:326-328) ...
        for st in self.data_store.values():
            st.clear()               # ... the kernel's reset does the same for the fused ones
        if mask is None:
            self.timestep = 0
        return self._collect_obs(extra), infos

    # ---- queries (mujoco_parent.py:366-478, mujoco_rl.py:355-395)
    def get_sensor_data(self, agent=None):
        sd = self._batch.sensordata[:, :self.model.nsensordata]
        if agent is not None:
            sd = sd[:, self.agents_observation_index[agent]["sensors"]]
        return self._out(sd)

    def get_observations(self, agent):
        b = self._batch
        oi = self.agents_observation_index[agent]
        o = torch.cat([b.sensordata[:, oi["sensors"]], b.qpos[:, oi["qpos"]], b.qvel[:, oi["qvel"]]], dim=1)
        return self._out(o)

    def get_camera_data(self, cam_object):
        """mujoco_parent.py:540-556: images of all cameras of an agent ([N, n_cams, H, W, 3] u8), or of one named
        camera ([N, H, W, 3]); num_envs = 1 returns the reference's numpy shapes.  Rows are bottom-up, as the
        reference's glReadPixels buffer.  Needs "agentCameras": True, like the reference."""
        if not self.agent_cameras:
            raise Exception("get_camera_data needs config 'agentCameras': True")
        w, h = self.sensor_resolution
        if cam_object in self._tables.rgb_sensors:
            names, squeeze = self._tables.rgb_sensors[cam_object], False
        else:
            names, squeeze = [cam_object], True
        ids = []
        for name in names:
            cid = self.model.name2id(L.OBJ_CAMERA, name)
            if cid < 0:
                raise KeyError(f"Invalid name '{name}'. Valid names: "
                               f"{[n for v in self._tables.rgb_sensors.values() for n in v]}")
            ids.append(cid)
        if not ids:
            img = torch.zeros((self.num_envs, 0, h, w, 3), dtype=torch.uint8, device=self.device)
        elif len(self._levels) == 1:
            img = self._batch.render(ids, w, h)
        else:   # every level renders all envs' qpos with its own geometry / colours; keep each env's own level
            img = self._levels[0]["batch"].render(ids, w, h)
            for lid, lv in enumerate(self._levels[1:], 1):
                sel = self.level_id == lid
                if bool(sel.any()):
                    img[sel] = lv["batch"].render(ids, w, h)[sel]
        if squeeze:
            img = img[:, 0]
        return img if self.num_envs > 1 else img[0].cpu().numpy()

    def get_camera_images(self, cam_object, depth=True, segmentation=True, final=False):
        """get_camera_data with more channels: a dict with `rgb` (u8 [N, n_cams, H, W, 3]), and on request `depth` (f32
        [N, n_cams, H, W], metres along the camera's optical axis, 0 where nothing is hit) and `segmentation` (i32
        [N, n_cams, H, W], MuJoCo geom id, -1 where nothing is hit), all from the same ray and hit (include/mjb.h,
        mjb_render_ex).  Agents, camera names, squeezing and num_envs = 1 as in get_camera_data.

        `final=True` (needs `autoReset`): the last frame of the episodes the last step() ended, rendered from the state
        their `final_observation` describes; the images of other envs are zero, and the dict also holds `mask` (bool [N],
        the last step's `_final_observation`)."""
        if not self.agent_cameras:
            raise Exception("get_camera_images needs config 'agentCameras': True")
        if final and not self.auto_reset:
            raise Exception("get_camera_images(final=True) needs config 'autoReset': True (without it no step ends an "
                            "episode inside the kernel, and the last state of every episode is the current one)")
        w, h = self.sensor_resolution
        names, squeeze = self.__camera_names(cam_object)
        ids = [self.__camera_id(n) for n in names]
        N = self.num_envs
        chans = dict(rgb=True, depth=bool(depth), segmentation=bool(segmentation))
        mask = None
        if final:
            A = len(self.agents)
            mask = (self._batch.term[:, A] | self._batch.trunc[:, A]).view(torch.bool).clone()
        if not ids:
            shapes = {"rgb": ((N, 0, h, w, 3), torch.uint8), "depth": ((N, 0, h, w), torch.float32),
                      "segmentation": ((N, 0, h, w), torch.int32)}
            out = {k: torch.zeros(shapes[k][0], dtype=shapes[k][1], device=self.device) for k, on in chans.items() if on}
        elif len(self._levels) == 1:
            out = self._batch.render_ex(ids, w, h, final=final, mask=mask, **chans)
        else:   # as get_camera_data: each env keeps the geometry / colours of its own level (no autoReset here, so no final)
            out = self._levels[0]["batch"].render_ex(ids, w, h, **chans)
            for lid, lv in enumerate(self._levels[1:], 1):
                sel = self.level_id == lid
                if bool(sel.any()):
                    other = lv["batch"].render_ex(ids, w, h, **chans)
                    for k in out:
                        out[k][sel] = other[k][sel]
        if squeeze:
            out = {k: v[:, 0] for k, v in out.items()}
        if N == 1:
            out = {k: v[0].cpu().numpy() for k, v in out.items()}
        if final:
            out["mask"] = mask if N > 1 else bool(mask[0].item())
        return out

    def __camera_names(self, cam_object):
        """(camera names, squeeze): all cameras of an agent, or one named camera"""
        if cam_object in self._tables.rgb_sensors:
            return self._tables.rgb_sensors[cam_object], False
        return [cam_object], True

    def __camera_id(self, name):
        cid = self.model.name2id(L.OBJ_CAMERA, name)
        if cid < 0:
            raise KeyError(f"Invalid name '{name}'. Valid names: {[n for v in self._tables.rgb_sensors.values() for n in v]}")
        return cid

    def _position(self, name_or_xyz):
        """[N, 3] position: exported probe, constant of a static object, or explicit coordinates"""
        if isinstance(name_or_xyz, str):
            name = name_or_xyz
            if name in self._probe_names:
                return self._batch.probe[:, self._probe_names.index(name), :3]
            ot, oid = self._resolve(name)
            sp = static_pose(self.model.fields, ot, oid)
            if sp is None:
                raise Exception(f"'{name}' moves and its position is not exported (exported: {self._probe_names}); "
                                f"add it to config_dict['exportPositions'] (or use \"all\")")
            return torch.tensor(sp[0], dtype=torch.float32, device=self.device).reshape(1, 3).expand(self.num_envs, 3)
        return torch.as_tensor(np.asarray(name_or_xyz, dtype=np.float32), device=self.device).reshape(-1, 3)

    def _orientation_quat(self, name):
        """[N, 4] (w, x, y, z) of the body frame (data.body(n).xmat) or geom frame (data.geom(n).xmat)"""
        ot, oid = self._resolve(name)
        sp = static_pose(self.model.fields, ot, oid)
        if sp is not None:
            return torch.tensor(sp[1], dtype=torch.float32, device=self.device).reshape(1, 4).expand(self.num_envs, 4)
        if name in self._probe_names and self._batch.buf.get("probe_quat") is not None:
            return self._batch.probe_quat[:, self._probe_names.index(name)]
        raise Exception(f"orientation of '{name}' is not exported: set config_dict['exportOrientation'] = True"
                        + ("" if name in self._probe_names else " and add it to config_dict['exportPositions']"))

    def distance(self, object_1, object_2):
        """mujoco_parent.py:428-449 (math.dist on float64 views): fp64 arithmetic on the fp32 positions"""
        v = self._position(object_1).double() - self._position(object_2).double()
        d = ((v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1]) + v[:, 2] * v[:, 2]).sqrt()
        return d if self.num_envs > 1 else d[0].item()

    def collision(self, geom_1, geom_2):
        def gid(g):
            if isinstance(g, str):
                i = self.model.name2id(L.OBJ_GEOM, g)
                if i < 0:
                    raise Exception(f"Collision object {g} not found in data")
                return i
            return int(g)
        g1, g2 = gid(geom_1), gid(geom_2)
        b = self._batch
        cg = b.contact_geom
        valid = torch.arange(cg.shape[1], device=self.device)[None, :] < b.ncon[:, None]
        hit = ((cg[:, :, 0] == g1) & (cg[:, :, 1] == g2)) | ((cg[:, :, 0] == g2) & (cg[:, :, 1] == g1))
        r = (hit & valid).any(dim=1)
        return r if self.num_envs > 1 else bool(r[0].item())

    def get_data(self, name):
        """mujoco_parent.py:394-426 + mujoco_rl.py:380-395.  `orientation` = zyx Euler angles in degrees of the body /
        geom frame (helper.py:6-18); None when the object moves and orientations are not exported."""
        ot, oid = self._resolve(name)
        f = self.model.fields
        pos = self._out(self._position(name))
        try:
            ori = self._out(quat_to_euler_zyx_deg(self._orientation_quat(name)))
        except Exception:
            ori = None
        if ot == L.OBJ_BODY:
            data = {"position": pos, "mass": np.array([f["body_mass"][oid]]) if self.num_envs == 1 else float(f["body_mass"][oid]),
                    "orientation": ori, "id": oid, "name": name, "type": "body"}
        else:
            data = {"position": pos, "orientation": ori, "id": oid, "name": name, "type": "geom",
                    "color": f["geom_rgba"][4 * oid:4 * oid + 4].astype(np.float32), "shape": int(f["geom_type"][oid])}
        if name in self.info_name_list:
            for key, val in self.info_json["environment"]["objects"][name].items():
                if key not in ["position", "orientation", "mass"]:
                    data[key] = val
        return data

    def filter_by_tag(self, tag):
        return [self.get_data(n) for n in self.__filter_names(tag)]

    # ---- raw device views for policy code
    @property
    def batch(self):
        return self._batch
