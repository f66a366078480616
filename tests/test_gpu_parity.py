"""Parity tests proper: the CUDA path through the C-ABI (libmjb.so) against the fp64 oracle.
Tolerance (BASELINE.json north_star: "about 1e-4 against MuJoCo fp64"): after ONE step from identical
states |x_gpu - x_ref| <= 1e-4 * max(1, |x_ref|) for qpos / qvel / sensordata; contact-pair sets,
Language observations, termination / truncation flags and drawn targets are compared EXACTLY.
Short-horizon drift bound: after 200 free-running steps |qpos_gpu - qpos_ref|_inf <= 5e-3 while no
contact event is missed (contact-rich trajectories are chaotic beyond that)."""
import os

import numpy as np
import pytest
import torch

from common import load_scene, make_spec, oracle_states
from mujoco_rl_environment_wrapper_b200 import _lib as L
from oracle import OracleSim
from oracle import host_loop as H

pytestmark = pytest.mark.gpu
RTOL = 1e-4


def rel_err(x, ref):
    return float((np.abs(x - ref) / np.maximum(1.0, np.abs(ref))).max()) if len(ref) else 0.0


def _batch(model, spec, n, keep):
    from mujoco_rl_environment_wrapper_b200.batch import Batch
    return Batch(model, spec, n, keepalive=keep)


def _upload(b, states, model, n_phys):
    nq, nv, nu = model.nq, model.nv, model.nu
    b.qpos[:len(states), :nq] = torch.tensor(np.stack([s[0][0] for s in states]), dtype=torch.float32)
    b.qvel[:len(states), :nv] = torch.tensor(np.stack([s[0][1] for s in states]), dtype=torch.float32)
    b.warmstart[:len(states), :nv] = torch.tensor(np.stack([s[0][2] for s in states]), dtype=torch.float32)
    if nu:
        b.ctrl[:len(states), :nu] = torch.tensor(np.stack([s[0][3] for s in states]), dtype=torch.float32)
    b.actions[:len(states), :, :n_phys] = torch.tensor(np.stack([s[0][4] for s in states]), dtype=torch.float32)


@pytest.mark.parametrize("scene,n,stride,settle", [("2A", 192, 6, 100), ("C1", 64, 8, 100), ("1A", 64, 6, 30),
                                                   ("S1", 32, 10, 50), ("S2", 32, 10, 50), ("S3", 32, 10, 50),
                                                   ("S4", 32, 10, 50), ("3S", 48, 10, 100)])
def test_one_step_parity(scene, n, stride, settle):
    model, tables, agents, fj = load_scene(scene)
    spec, keep = make_spec(model, tables, agents, fj)
    states = oracle_states(model, tables, agents, fj, n, stride=stride, settle=settle, seed=3)
    b = _batch(model, spec, len(states), keep)
    _upload(b, states, model, spec.n_phys_act)
    b.physics(1)
    b.sync()
    q, v, sd = b.qpos.cpu().numpy(), b.qvel.cpu().numpy(), b.sensordata.cpu().numpy()
    ncon, cg = b.ncon.cpu().numpy(), b.contact_geom.cpu().numpy()
    ns = model.nsensordata
    total = 0
    for e, (pre, post) in enumerate(states):
        assert rel_err(q[e, :model.nq], post["qpos"]) < RTOL, (scene, e)
        assert rel_err(v[e, :model.nv], post["qvel"]) < RTOL, (scene, e)
        if ns:
            # acceleration-stage sensors (touch, accelerometer) are O(qacc), not O(h * qacc) like the state:
            # fp32 contact forces on redundant contacts carry ~1e-4..1e-3 relative noise
            tol = 2e-3 if scene in ("S1", "S2", "3S") else RTOL
            assert rel_err(sd[e, :ns], post["sensordata"][:ns]) < tol, (scene, e)
        assert sorted((int(a), int(c)) for a, c in cg[e, :ncon[e]]) == post["pairs"], (scene, e)
        total += ncon[e]
    assert total > 0


def test_short_horizon_drift_2A():
    model, tables, agents, fj = load_scene("2A")
    spec, keep = make_spec(model, tables, agents, fj)
    b = _batch(model, spec, 8, keep)
    b.reset(); b.sync()
    sims = [OracleSim(model.blob) for _ in range(8)]
    rng = np.random.default_rng(5)
    idx = np.array(tables.agents_action_index["sender"] + tables.agents_action_index["receiver"])
    for t in range(200):
        act = rng.uniform(-1, 1, (8, 2, 8)).astype(np.float32)
        b.actions[:, :, :8] = torch.tensor(act)
        b.physics(1)
        for e, s in enumerate(sims):
            s.ctrl[idx] = act[e].reshape(-1)
            s.step()
    b.sync()
    q = b.qpos.cpu().numpy()
    for e, s in enumerate(sims):
        assert np.abs(q[e, :30] - s.qpos).max() < 5e-3


def _resolver(model):
    def resolve(name):
        bid = model.name2id(L.OBJ_BODY, name)
        return (1, bid) if bid >= 0 else (5, model.name2id(L.OBJ_GEOM, name))
    return resolve


def test_full_step_C2_flags_bit_exact():
    """Config C2 through the drop-in class: Language + tag-distance reward + done on 64 envs, each env
    mirrored by one reference-order host loop on the oracle; states re-synchronised every step."""
    import os
    from common import LEVELS
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    N, seed, max_steps = 64, 4321, 7
    env = MuJoCoRL({"xmlPath": os.path.join(LEVELS, "two_ants.xml"), "infoJson": os.path.join(LEVELS, "info_2A.json"),
                    "agents": ["sender", "receiver"], "skipFrames": 1, "maxSteps": max_steps, "num_envs": N, "seed": seed,
                    "environmentDynamics": [P.Language], "rewardFunctions": [P.tag_distance_reward],
                    "doneFunctions": [P.distance_done]})
    model, tables, agents = env.model, env._tables, env.agents
    lib = L.load()
    mirrors = [H.OracleEnv(model, tables, agents, max_steps=max_steps, dynamics=[H.Language],
                           reward_functions=[H.tag_distance_reward], done_functions=[H.distance_done],
                           targets=["choice_1", "choice_2"], draw=(lambda e: lambda a, k: lib.mjb_draw_u32(seed, e, a, k))(e),
                           resolve=_resolver(model)) for e in range(N)]
    obs, infos = env.reset()
    act0 = env.batch.actions[:, :, :9].cpu().numpy()
    for e, m in enumerate(mirrors):
        o, _ = m.reset({a: act0[e, i] for i, a in enumerate(agents)})
        for i, a in enumerate(agents):
            assert rel_err(obs[a][e].cpu().numpy(), o[a]) < RTOL
    assert env.observation_space("sender").shape == (60,) and env.action_space("sender").shape == (9,)
    rng = np.random.default_rng(2)
    b = env.batch
    for t in range(10):
        act = np.concatenate([rng.uniform(-1, 1, (N, 2, 8)), rng.uniform(0, 3, (N, 2, 1))], axis=2).astype(np.float32)
        # random restarts of a few envs far from / close to a target so that done flags flip
        for e, m in enumerate(mirrors):
            if t == 3 and e % 4 == 0:
                m.sim.qpos[0:2] = [7.0, -2.0] if e % 8 == 0 else [1.4, -2.1]
                m.sim.qpos[2] = 1.25
        b.qpos[:, :30] = torch.tensor(np.stack([m.sim.qpos for m in mirrors]), dtype=torch.float32)
        b.qvel[:, :28] = torch.tensor(np.stack([m.sim.qvel for m in mirrors]), dtype=torch.float32)
        b.warmstart[:, :28] = torch.tensor(np.stack([m.sim.qacc_warmstart for m in mirrors]), dtype=torch.float32)
        o, r, term, trunc, info = env.step({a: torch.tensor(act[:, i]) for i, a in enumerate(agents)})
        flips = 0
        for e, m in enumerate(mirrors):
            mo, mr, mterm, mtrunc, _ = m.step({a: act[e, i] for i, a in enumerate(agents)})
            for i, a in enumerate(agents):
                assert rel_err(o[a][e].cpu().numpy()[:59], mo[a][:59]) < RTOL, (t, e, a)
                assert o[a][e, 59].item() == mo[a][59]
                assert abs(r[a][e].item() - mr[a]) < 2e-3
                assert bool(term[a][e]) == mterm[a] and bool(trunc[a][e]) == mtrunc[a], (t, e, a)
            assert bool(term["__all__"][e]) == mterm["__all__"] and bool(trunc["__all__"][e]) == mtrunc["__all__"]
            flips += mterm["__all__"]
        if t >= 3:
            assert flips > 0
    assert set(info["sender"].keys()) == {"Language"}


def test_full_size_properties():
    """BASELINE sizes (65536 envs): run-to-run bit-reproducibility, env-index independence (identical envs
    with identical actions stay bit-identical wherever they sit in the grid) and reset idempotence."""
    model, tables, agents, fj = load_scene("2A")
    spec, keep = make_spec(model, tables, agents, fj)
    N = 65536
    b = _batch(model, spec, N, keep)
    g = torch.Generator(device="cuda"); g.manual_seed(0)
    acts = torch.rand((6, 1, 2, 8), generator=g, device="cuda") * 2 - 1
    outs = []
    for rep in range(2):
        b.reset(); 
        for k in range(6):
            b.actions[:, :, :8] = acts[k]
            b.physics(1)
        b.sync()
        outs.append((b.qpos.clone(), b.qvel.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    assert bool((outs[0][0] == outs[0][0][0:1]).all()) and bool((outs[0][1] == outs[0][1][0:1]).all())
    assert bool(torch.isfinite(outs[0][0]).all())
    # contact slots: a 400-step random rollout of 65536 envs never fills the per-env contact table
    g2 = torch.Generator(device="cuda"); g2.manual_seed(1)
    worst = 0
    for k in range(400):
        b.actions[:, :, :8] = torch.rand((N, 2, 8), generator=g2, device="cuda") * 2 - 1
        b.physics(1)
        if k % 20 == 19:
            worst = max(worst, int(b.ncon.max()))
    assert 0 < worst < b.layout.maxcon, worst
    assert bool(torch.isfinite(b.qpos).all()) and bool(torch.isfinite(b.qvel).all())
    b.reset(); b.sync(); q1 = b.qpos.clone(); b.reset(); b.sync()
    assert torch.equal(q1, b.qpos)
    mask = torch.zeros(N, dtype=torch.uint8, device="cuda"); mask[::2] = 1
    b.actions[:, :, :8] = acts[0]; b.physics(3); b.reset(mask); b.sync()
    assert torch.equal(b.qpos[::2], q1[::2]) and not torch.equal(b.qpos[1::2], q1[1::2])


def test_literal_skipframes0_freejoint():
    """The reference benchmarks' literal configuration (skipFrames = 0, freeJoint = True): no physics,
    qvel overwrite + observation gather only (SURVEY A.4 Q1)."""
    model, tables, agents, fj = load_scene("1A")
    from mujoco_rl_environment_wrapper_b200.tables import Tables
    import os
    from common import LEVELS
    text = open(os.path.join(LEVELS, "ant_rk4.xml")).read()
    tables = Tables(text, model, agents, True)
    spec, keep = make_spec(model, tables, agents, True, skip_frames=0, rewards=[(L.REW_ANT, 0.0)])
    b = _batch(model, spec, 128, keep)
    b.reset(); b.sync()
    q0 = b.qpos.clone()
    a = torch.rand((128, 1, 3), device="cuda") * 2 - 1
    b.actions[:, :, :3] = a
    b.step(); b.sync()
    assert torch.equal(b.qpos, q0)
    assert torch.equal(b.qvel[:, [0, 1, 5]], a[:, 0])
    assert torch.equal(b.obs[:, 0, 15:15 + 14], b.qvel[:, :14])
    assert float(b.reward.abs().max()) == 0.0 and int(b.timestep[0]) == 1


def test_no_cpu_fallback_symbols_loaded():
    """The product library is the thing that ran: kernel launches were counted by the handle."""
    model, tables, agents, fj = load_scene("S3")
    spec, keep = make_spec(model, tables, agents, fj)
    b = _batch(model, spec, 16, keep)
    n0 = b.launch_count
    b.reset(); b.physics(2); b.forward(); b.sync()
    assert b.launch_count == n0 + 3


def _mirror_env(env, e, seed, dynamics, rewards, dones, targets, **kw):
    lib = L.load()
    return H.OracleEnv(env.model, env._tables, env.agents, dynamics=dynamics, reward_functions=rewards, done_functions=dones,
                       targets=targets, draw=(lambda a, k: lib.mjb_draw_u32(seed, e, a, k)), resolve=_resolver(env.model), **kw)


def _sync_state(env, mirrors):
    b, m = env.batch, env.model
    b.qpos[:, :m.nq] = torch.tensor(np.stack([x.sim.qpos for x in mirrors]), dtype=torch.float32)
    b.qvel[:, :m.nv] = torch.tensor(np.stack([x.sim.qvel for x in mirrors]), dtype=torch.float32)
    if m.nu:
        b.ctrl[:, :m.nu] = torch.tensor(np.stack([x.sim.ctrl for x in mirrors]), dtype=torch.float32)


def test_pick_up_dynamic_C5():
    """Config C5: Pick_Up dynamic re-expressed per agent (Testing/Pick_Up_Dynamic.py, SURVEY a9): inventory toggles,
    target re-draws and the 4 appended observations, against the reference-order host loop on identical draws."""
    import os
    from common import LEVELS
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    N, seed = 32, 77
    env = MuJoCoRL({"xmlPath": os.path.join(LEVELS, "two_ants.xml"), "infoJson": os.path.join(LEVELS, "info_2A.json"),
                    "agents": ["sender", "receiver"], "num_envs": N, "seed": seed, "environmentDynamics": [P.PickUpDynamic]})
    assert env.observation_space("sender").shape == (63,) and env.action_space("sender").shape == (8,)
    mirrors = [_mirror_env(env, e, seed, [H.PickUp], [], [], ["choice_1", "choice_2"]) for e in range(N)]
    env.reset()
    for m in mirrors:
        m.reset({a: np.zeros(8) for a in env.agents})
    rng = np.random.default_rng(9)
    toggles = 0
    for t in range(8):
        for e, m in enumerate(mirrors):
            if t in (2, 5) and e % 2 == 0:           # drop the sender next to a target (distance < 2 -> pick up)
                m.sim.qpos[0:3] = [6.0, -1.5, 1.3] if (e // 2) % 2 == 0 else [1.0, -1.2, 1.3]
        _sync_state(env, mirrors)
        act = rng.uniform(-1, 1, (N, 2, 8)).astype(np.float32)
        o, r, term, trunc, info = env.step({a: torch.tensor(act[:, i]) for i, a in enumerate(env.agents)})
        for e, m in enumerate(mirrors):
            mo, mr, mterm, mtrunc, _ = m.step({a: act[e, i] for i, a in enumerate(env.agents)})
            for i, a in enumerate(env.agents):
                g = o[a][e].cpu().numpy()
                assert rel_err(g[:59], mo[a][:59]) < RTOL
                assert np.allclose(g[59:62], mo[a][59:62], atol=1e-5)          # target position
                assert g[62] == mo[a][62]                                        # inventory, exact
                assert r[a][e].item() == mr[a]                                   # 0 / 1, exact
                toggles += int(mr[a])
    assert toggles > 0
    assert set(info["sender"].keys()) == {"PickUpDynamic"}


def test_ant_reward_rk4_C3_and_skipframes():
    """Config C3 physics-on: Ant.xml (RK4, dt 0.01), ant_reward_function, skipFrames = 5 (ant_learning_perf.py:51-53)."""
    import os
    from common import LEVELS
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    N = 16
    env = MuJoCoRL({"xmlPath": os.path.join(LEVELS, "ant_rk4.xml"), "agents": ["torso"], "num_envs": N, "skipFrames": 5,
                    "rewardFunctions": [P.ant_reward_function], "maxSteps": 3})
    mirrors = [_mirror_env(env, e, 0, [], [H.ant_reward], [], [], skip_frames=5, max_steps=3) for e in range(N)]
    env.reset()
    for m in mirrors:
        m.reset({"torso": np.zeros(8)})
    rng = np.random.default_rng(4)
    for t in range(6):
        _sync_state(env, mirrors)
        act = rng.uniform(-1, 1, (N, 1, 8)).astype(np.float32)
        o, r, term, trunc, info = env.step({"torso": torch.tensor(act[:, 0])})
        for e, m in enumerate(mirrors):
            mo, mr, mterm, mtrunc, _ = m.step({"torso": act[e, 0]})
            assert rel_err(o["torso"][e].cpu().numpy(), mo["torso"]) < 5 * RTOL      # 5 RK4 substeps
            assert abs(r["torso"][e].item() - mr["torso"]) < 2e-2 * max(1.0, abs(mr["torso"]))  # (dx / dt) amplifies fp32 by 100
            assert bool(trunc["torso"][e]) == mtrunc["torso"] and bool(trunc["__all__"][e]) == mtrunc["__all__"]
        assert "__all__" not in term                # no done function configured (SURVEY 3.3)


def test_sensor_scene_C4_skipframes5_freejoint():
    """Config C4: 3-sensor level, freeJoint actions, skipFrames = 5 (sensor_test.py:18-20)."""
    model, tables, agents, fj = load_scene("3S")
    spec, keep = make_spec(model, tables, agents, fj, skip_frames=5)
    N = 24
    b = _batch(model, spec, N, keep)
    b.reset(); b.sync()
    sims = [OracleSim(model.blob) for _ in range(N)]
    for s in sims:
        s.forward()
    rng = np.random.default_rng(8)
    idx = tables.agents_action_index["sender"] + tables.agents_action_index["receiver"]
    for t in range(30):
        act = rng.uniform(-1, 1, (N, 2, 3)).astype(np.float32)
        b.qpos[:, :30] = torch.tensor(np.stack([s.qpos for s in sims]), dtype=torch.float32)
        b.qvel[:, :28] = torch.tensor(np.stack([s.qvel for s in sims]), dtype=torch.float32)
        b.actions[:, :, :3] = torch.tensor(act)
        b.step(); b.sync()
        obs = b.obs.cpu().numpy()
        for e, s in enumerate(sims):
            s.qvel[idx] = act[e].reshape(-1)
            for _ in range(5):
                s.step()
            for i, a in enumerate(agents):
                oi = tables.agents_observation_index[a]
                ref = np.concatenate([s.sensordata[oi["sensors"]], s.qpos, s.qvel])
                assert rel_err(obs[e, i, :63][5:], ref[5:]) < 5 * RTOL, (t, e)
                assert rel_err(obs[e, i, :5], ref[:5]) < 5e-3, (t, e, obs[e, i, :5], ref[:5])


def test_single_env_squeezes_to_reference_shapes_and_wrappers():
    """num_envs = 1 (the reference's only mode): numpy float64 observations, Python scalars, dict keys as the
    reference returns them; the Gymnasium / Gym adapters on top (wrappers.py:12-142)."""
    import os
    from common import LEVELS
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    from mujoco_rl_environment_wrapper_b200.wrappers import GymnasiumWrapper, GymWrapper
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    env = MuJoCoRL({"xmlPath": os.path.join(LEVELS, "ant_rk4.xml"), "agents": ["torso"], "maxSteps": 2,
                    "rewardFunctions": [P.ant_reward_function]})
    obs, infos = env.reset()
    assert isinstance(obs["torso"], np.ndarray) and obs["torso"].dtype == np.float64 and obs["torso"].shape == (29,)
    o, r, term, trunc, info = env.step({"torso": env.action_space("torso").sample()})
    assert isinstance(r["torso"], float) and term == {"torso": False} and trunc == {"torso": False, "__all__": False}
    assert info == {"torso": {}}
    env.step({"torso": np.zeros(8, np.float32)})
    *_, trunc, _ = env.step({"torso": np.zeros(8, np.float32)})
    assert trunc["__all__"] is True                       # third call with maxSteps = 2
    g = GymnasiumWrapper(env, "torso")
    o, info = g.reset()
    o, r, term, trunc, info = g.step(g.action_space.sample())
    assert o.shape == (29,) and isinstance(term, bool) and trunc is False
    o, r, done, info = GymWrapper(env, "torso").step(np.zeros(8, np.float32))
    assert done is False
    with pytest.raises(Exception, match="too many agents"):
        two = MuJoCoRL({"xmlPath": os.path.join(LEVELS, "two_ants.xml"), "agents": ["sender", "receiver"]})
        GymnasiumWrapper(two, "sender")


def test_user_plugins_run_as_batched_torch_code():
    """Unknown plugins keep the reference's signatures (`dynamic(agent, actions)`, `f(env, agent)`) and run as
    batched torch code after the kernel; fused and user plugins can be mixed."""
    import os
    from common import LEVELS
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    from mujoco_rl_environment_wrapper_b200 import plugins as P

    class Echo:
        def __init__(self, mujoco_gym):
            self.mujoco_gym = mujoco_gym
            self.observation_space = {"low": [-5, -5], "high": [5, 5]}
            self.action_space = {"low": [-1, -1], "high": [1, 1]}

        def dynamic(self, agent, actions):
            env = self.mujoco_gym
            a = torch.as_tensor(actions, dtype=torch.float32, device=env.device).reshape(env.num_envs, 2)
            env.data_store[agent]["last"] = a
            return a.sum(dim=1), 2 * a, a[:, 0] > 0.9, {"who": agent}

    def height_reward(env, agent):
        return env.batch.qpos[:, 2] if agent == "sender" else env.batch.qpos[:, 17]

    def never_done(env, agent):
        return torch.zeros(env.num_envs, dtype=torch.bool, device=env.device)

    N = 8
    env = MuJoCoRL({"xmlPath": os.path.join(LEVELS, "two_ants.xml"), "agents": ["sender", "receiver"], "num_envs": N,
                    "environmentDynamics": [P.Language, Echo], "rewardFunctions": [height_reward], "doneFunctions": [never_done]})
    assert env.action_routing["dynamic"] == {"Language": [8, 9], "Echo": [9, 11]}
    assert env.observation_space("sender").shape == (62,) and env.action_space("sender").shape == (11,)
    env.reset()
    act = torch.rand(N, 2, 11, device="cuda") * 2 - 1
    act[:, :, 8] = torch.tensor([1.7, 2.2], device="cuda")
    o, r, term, trunc, info = env.step(act)
    assert o["sender"].shape == (N, 62)
    assert torch.equal(o["sender"][:, 59], torch.zeros(N, device="cuda")) and torch.equal(o["receiver"][:, 59], torch.ones(N, device="cuda"))
    assert torch.allclose(o["sender"][:, 60:62], 2 * act[:, 0, 9:11])
    assert torch.allclose(r["sender"], act[:, 0, 9:11].sum(1) + env.batch.qpos[:, 2])
    assert torch.equal(term["receiver"], act[:, 1, 9] > 0.9) and "__all__" in term
    assert info["sender"]["Echo"] == {"who": "sender"} and info["sender"]["Language"] == {}
    assert torch.equal(env.data_store["sender"]["last"], act[:, 0, 9:11])
    assert torch.equal(env.data_store["receiver"]["utterance"], torch.full((N,), 2, dtype=torch.int32, device="cuda"))


def test_queries_distance_collision_get_data_filter_by_tag():
    """mujoco_parent.py:394-478 / mujoco_rl.py:355-395 on the batched env."""
    import os
    from common import LEVELS
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    N = 16
    env = MuJoCoRL({"xmlPath": os.path.join(LEVELS, "two_ants.xml"), "infoJson": os.path.join(LEVELS, "info_2A.json"),
                    "agents": ["sender", "receiver"], "num_envs": N})
    env.reset()
    tg = env.filter_by_tag("target")
    assert [t["name"] for t in tg] == ["choice_1", "choice_2"] and tg[0]["type"] == "body" and tg[0]["tags"] == ["target"]
    d = env.distance("sender", "choice_1")
    ref = np.linalg.norm(np.array([-5.522553, 0.9194446, 1.0]) - np.array([7.02852, -2.071592, 0.4710507]))
    assert d.dtype == torch.float64   # the reference's distance is math.dist on float64 views (mujoco_parent.py:449)
    assert torch.allclose(d, torch.full((N,), ref, device="cuda", dtype=torch.float64), rtol=1e-5)
    assert not bool(env.collision("sender_geom", "choice_1_geom").any())
    for _ in range(400):
        env.step({a: torch.zeros(N, 8) for a in env.agents})
    # settled: some ankle capsule of every ant touches the floor (geom 0 is the unnamed plane)
    touching = torch.zeros(N, dtype=torch.bool, device="cuda")
    for g in ("left_ankle_geom", "right_ankle_geom", "third_ankle_geom", "fourth_ankle_geom"):
        touching |= env.collision(0, g)
    assert bool(touching.all())
    with pytest.raises(Exception, match="not found"):
        env.collision("nope", "sender_geom")
    assert env.get_data("sender")["mass"] == pytest.approx(5.0 * 4 / 3 * np.pi * 0.25 ** 3)
    with pytest.raises(KeyError):
        env.get_data("no_such_object")


def test_inter_ant_contacts_couple_the_trees():
    """Two ants dropped onto each other: contacts between the two kinematic trees make the Newton Hessian a
    single 28 x 28 block (shared-memory factorisation path instead of the per-tree register path) and exercise
    capsule-capsule / sphere-capsule pairs across agents.  One step from identical states vs the oracle."""
    model, tables, agents, fj = load_scene("2A")
    spec, keep = make_spec(model, tables, agents, fj)
    sim = OracleSim(model.blob)
    rng = np.random.default_rng(21)
    idx = np.array(tables.agents_action_index["sender"] + tables.agents_action_index["receiver"])
    states, cross = [], 0
    geom_body = model.fields["geom_bodyid"]
    root = model.fields["body_rootid"]
    for trial in range(24):
        sim.reset()
        # receiver straight above the sender, slightly offset and yawed, then let them fall together
        sim.qpos[15:18] = sim.qpos[0:3] + np.array([rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3), 0.45 + 0.2 * rng.random()])
        yaw = rng.uniform(0, np.pi)
        sim.qpos[18:22] = [np.cos(yaw / 2), 0, 0, np.sin(yaw / 2)]
        for t in range(260):
            c = rng.uniform(-1, 1, 16)
            sim.ctrl[idx] = c
            if t >= 60 and t % 10 == 0:
                pre = (sim.qpos.copy(), sim.qvel.copy(), sim.qacc_warmstart.copy(), sim.ctrl.copy(), c.reshape(2, 8).copy())
                sim.step()
                pairs = sim.contact_pairs()
                ncross = sum(1 for a, b in pairs if root[geom_body[a]] != root[geom_body[b]] and root[geom_body[a]] and root[geom_body[b]])
                cross += ncross > 0
                states.append((pre, {"qpos": sim.qpos.copy(), "qvel": sim.qvel.copy(), "pairs": sorted(pairs)}))
            else:
                sim.step()
    assert cross > 40, cross          # the sample really contains inter-tree contacts
    b = _batch(model, spec, len(states), keep)
    _upload(b, states, model, 8)
    b.physics(1); b.sync()
    q, v = b.qpos.cpu().numpy(), b.qvel.cpu().numpy()
    ncon, cg = b.ncon.cpu().numpy(), b.contact_geom.cpu().numpy()
    assert int(ncon.max()) < b.layout.maxcon
    for e, (pre, post) in enumerate(states):
        assert rel_err(q[e, :30], post["qpos"]) < RTOL, e
        assert rel_err(v[e, :28], post["qvel"]) < RTOL, e
        assert sorted((int(a), int(c_)) for a, c_ in cg[e, :ncon[e]]) == post["pairs"], e


# ---- SURVEY 8(f3): level variants (`xmlPath` list re-drawn at reset, mujoco_parent.py:88-91,351-356)
def _level_variants(tmp_path):
    """two structurally identical levels: B moves / shrinks the target boxes and names other targets"""
    import json
    import os
    lv = os.path.join(os.path.dirname(__file__), "levels")
    a = open(os.path.join(lv, "two_ants.xml")).read()
    b = a.replace('pos="7.02852 -2.071592 0.4710507"', 'pos="3.5 1.25 0.4710507"').replace(
        'size="1 1 0.5" rgba="255 0 0 1"', 'size="0.6 0.8 0.5" rgba="0 255 0 1"')
    assert a != b
    ja = json.load(open(os.path.join(lv, "info_2A.json")))
    jb = {"environment": {"objects": {"choice_1": {"tags": ["target"]}, "choice_2": {"tags": []},
                                      "reference": {"tags": ["target"]}}}, "areas": {}}
    paths = []
    for name, xml, js in (("LevelA", a, ja), ("LevelB", b, jb)):
        open(tmp_path / f"{name}.xml", "w").write(xml)
        json.dump(js, open(tmp_path / f"{name}.json", "w"))
        paths.append((str(tmp_path / f"{name}.xml"), str(tmp_path / f"{name}.json")))
    return paths


@pytest.mark.gpu
def test_level_variants_match_single_level_envs(tmp_path):
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    (xa, ja), (xb, jb) = _level_variants(tmp_path)
    N = 96
    common = dict(agents=["sender", "receiver"], environmentDynamics=[P.Language], rewardFunctions=[P.tag_distance_reward],
                  doneFunctions=[P.distance_done], num_envs=N, seed=7)
    multi = MuJoCoRL(dict(common, xmlPath=[xa, xb], infoJson=[ja, jb]))
    singles = [MuJoCoRL(dict(common, xmlPath=xa, infoJson=ja)), MuJoCoRL(dict(common, xmlPath=xb, infoJson=jb))]
    envs = [multi] + singles
    for e in envs:
        e.reset()
    lid = multi.level_id.cpu().numpy()
    assert set(lid.tolist()) == {0, 1}, "the draw must use both levels"

    def check(tag):
        for name in ("qpos", "qvel", "obs", "reward", "term", "trunc", "store_i", "store_f", "timestep"):
            got = getattr(multi.batch, name).cpu().numpy()
            want = np.where(lid.reshape((-1,) + (1,) * (got.ndim - 1)) == 0, getattr(singles[0].batch, name).cpu().numpy(),
                            getattr(singles[1].batch, name).cpu().numpy())
            # bit for bit (store_f carries an fp64 distance in two float columns: compare bytes, not float values)
            assert got.tobytes() == np.ascontiguousarray(want).tobytes(), f"{tag}: {name} differs from the single-level env of the same level"

    check("reset")
    for t in range(40):
        acts = [e.sample_actions() for e in envs]
        assert torch.equal(acts[0], acts[1]) and torch.equal(acts[0], acts[2])
        for e, a in zip(envs, acts):
            e.step(a)
        check(f"step {t}")
    # the two levels really differ (the moved box is where ants of level B collide / measure distances)
    assert singles[0].batch.store_f.cpu().numpy().tobytes() != singles[1].batch.store_f.cpu().numpy().tobytes()

    # masked reset: only the masked envs get a new level and a fresh state
    before = {k: getattr(multi.batch, k).clone() for k in ("qpos", "qvel", "timestep")}
    mask = torch.zeros(N, dtype=torch.bool)
    mask[::3] = True
    multi.reset(mask=mask)
    lid2 = multi.level_id.cpu().numpy()
    m = mask.numpy()
    assert np.array_equal(lid2[~m], lid[~m])
    assert (lid2[m] != lid[m]).any(), "some masked env should have moved to the other level"
    for k, v in before.items():
        assert torch.equal(getattr(multi.batch, k)[~mask], v[~mask]), f"{k} of unmasked envs must not change"
    assert int(multi.batch.timestep[mask].abs().sum()) == 0
    singles[0].reset()   # qpos0 is the same in both levels (only static boxes moved)
    assert torch.equal(multi.batch.qpos[mask], singles[0].batch.qpos[mask])
    for t in range(5):  # and the mixed batch keeps stepping
        multi.step(multi.sample_actions())
    assert torch.isfinite(multi.batch.qpos).all()


@pytest.mark.gpu
def test_level_variants_single_env_follows_reference_draw(tmp_path):
    """num_envs = 1: the level is random.choice(xmlPath) at construction and again at every reset, and the env's
    `xml_path`, `info_json`, `info_name_list` follow it (mujoco_parent.py:88-91,351-352; mujoco_rl.py:304-310)"""
    import random
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    (xa, ja), (xb, jb) = _level_variants(tmp_path)
    random.seed(3)
    expect = [random.choice([xa, xb]) for _ in range(7)]
    random.seed(3)
    env = MuJoCoRL({"xmlPath": [xa, xb], "infoJson": [ja, jb], "agents": ["sender", "receiver"]})
    seen = [env.xml_path]
    for _ in range(6):
        env.reset()
        seen.append(env.xml_path)
        want_tags = ["target"] if env.xml_path == xa else []
        assert env.info_json["environment"]["objects"]["choice_2"]["tags"] == want_tags
        obs, *_ = env.step({a: env.action_space(a).sample() for a in env.agents})
        assert obs["sender"].shape == (59,)
    assert seen == expect and len(set(seen)) == 2
    # a level that currently owns NO env must not step / reset the env with its model (an empty id list used to
    # reach the C side as NULL = "all envs": two steps per step(), obs from the wrong level)
    singles = {xa: MuJoCoRL({"xmlPath": xa, "infoJson": ja, "agents": ["sender", "receiver"]}),
               xb: MuJoCoRL({"xmlPath": xb, "infoJson": jb, "agents": ["sender", "receiver"]})}
    rng = np.random.default_rng(0)
    for _ in range(4):
        env.reset()
        ref = singles[env.xml_path]
        ref.reset()
        for t in range(6):
            act = {a: rng.uniform(-1, 1, 8).astype(np.float32) for a in env.agents}
            o1, *_ = env.step(act)
            o2, *_ = ref.step(act)
            assert int(env.batch.timestep[0]) == t + 1 == int(ref.batch.timestep[0])
            assert torch.equal(env.batch.qpos, ref.batch.qpos) and torch.equal(env.batch.qvel, ref.batch.qvel)
            assert np.array_equal(o1["sender"], o2["sender"]) and np.array_equal(o1["receiver"], o2["receiver"])


@pytest.mark.gpu
def test_level_variants_reject_structural_mismatch(tmp_path):
    import os
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    lv = os.path.join(os.path.dirname(__file__), "levels")
    with pytest.raises(Exception, match="structurally identical"):
        MuJoCoRL({"xmlPath": [os.path.join(lv, "two_ants.xml"), os.path.join(lv, "two_ants_touch.xml")],
                  "agents": ["sender", "receiver"], "num_envs": 4})


@pytest.mark.gpu
@pytest.mark.parametrize("scene_xml,agents,n,pinned", [
    ("two_ants.xml", ["sender", "receiver"], 100, True), ("two_ants.xml", ["sender", "receiver"], 3, True),
    ("two_ants.xml", ["sender", "receiver"], 37, False), ("one_ant_arena.xml", ["sender"], 101, True),
    ("one_ant_arena.xml", ["sender"], 3, True), ("one_ant_arena.xml", ["sender"], 101, False),
    ("ant_rk4.xml", ["torso"], 64, True), ("ant_rk4.xml", ["torso"], 64, False)])
def test_step_host_matches_device_step(scene_xml, agents, n, pinned):
    """mjb_step_host (host arrays in / out) returns exactly what mjb_step leaves in the device buffers: page-locked
    arrays written by the kernel itself (zero-copy; two launches on two streams from 4 envs per env-warp on, one below:
    n = 3), pageable arrays uploaded and copied back through the staging area; each also with several envs per warp
    (one_ant_arena, a ragged split at 101) and with the no-physics tile kernel (ant_rk4)."""
    import os
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    lv = os.path.join(os.path.dirname(__file__), "levels")
    cfg = {"xmlPath": os.path.join(lv, scene_xml), "agents": agents, "num_envs": n, "seed": 11}
    if len(agents) == 2:
        cfg.update(infoJson=os.path.join(lv, "info_2A.json"), environmentDynamics=[P.Language],
                   rewardFunctions=[P.tag_distance_reward], doneFunctions=[P.distance_done])
    if scene_xml == "ant_rk4.xml":
        cfg.update(freeJoint=True, skipFrames=0, rewardFunctions=[P.ant_reward_function])   # the no-physics step kernel
    dev, host = MuJoCoRL(cfg), MuJoCoRL(cfg)
    dev.reset(); host.reset()
    hb = host.batch
    arrs = hb.host_arrays(pinned=pinned)
    if not pinned:
        arrs = tuple(np.array(a) for a in arrs)   # plain pageable numpy
    h_act, h_obs, h_rew, h_term, h_trunc = arrs
    for t in range(25):
        a = dev.sample_actions()
        assert torch.equal(a, host.sample_actions())
        dev.batch.actions[:, :, :dev._act_dim] = a
        dev.batch.step()
        h_act[:, :, :dev._act_dim] = a.cpu().numpy()
        hb.step_host(h_act, h_obs, h_rew, h_term, h_trunc)
        for name, got in (("obs", h_obs), ("reward", h_rew), ("term", h_term), ("trunc", h_trunc)):
            assert np.array_equal(got, getattr(dev.batch, name).cpu().numpy()), (t, name)
        assert torch.equal(hb.qpos, dev.batch.qpos)


@pytest.mark.gpu
@pytest.mark.parametrize("xml,free_joint", [("two_ants_touch_acc.xml", False), ("two_ants_touch_acc.xml", True), ("box_rangefinder.xml", True)])
def test_parallel_api_conformance(xml, free_joint):
    """The checks of the reference's own API test (tests/parallel_env_test.py -> pettingzoo parallel_api_test) and of
    tests/sensor_test.py (observations stay inside the declared sensor bounds), restated without pettingzoo:
    stable space objects, dict keys = agents (+ "__all__" where the reference adds it), observations of the declared
    shape inside [low, high], numeric rewards, boolean flags, truncation from call maxSteps + 1 on (the reference's off-by-one)."""
    import os
    from common import LEVELS
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    two = xml.startswith("two_ants")
    agents = ["sender", "receiver"] if two else ["receiver"]
    cfg = {"xmlPath": os.path.join(LEVELS, xml), "agents": agents, "freeJoint": free_joint, "skipFrames": 5, "maxSteps": 40}
    if two:
        cfg.update(environmentDynamics=[P.Language], infoJson=os.path.join(LEVELS, "info_2A.json"),
                   rewardFunctions=[P.tag_distance_reward], doneFunctions=[P.distance_done])
    env = MuJoCoRL(cfg)
    assert env.agents == agents and env.possible_agents == agents
    for a in agents:
        assert env.observation_space(a) is env.observation_space(a) and env.action_space(a) is env.action_space(a)
    obs, infos = env.reset()
    assert set(obs) == set(agents) and set(infos) == set(agents)
    finite_bounds = 0
    for t in range(42):
        act = {a: env.action_space(a).sample() for a in agents}
        obs, rew, term, trunc, infos = env.step(act)
        assert set(obs) == set(rew) == set(infos) == set(agents)
        assert set(trunc) == set(agents) | {"__all__"}
        assert set(term) == (set(agents) | {"__all__"} if two else set(agents))   # "__all__" only with done functions
        for a in agents:
            sp = env.observation_space(a)
            assert obs[a].shape == sp.low.shape and np.isfinite(obs[a]).all()
            assert (obs[a] >= sp.low - 1e-6).all() and (obs[a] <= sp.high + 1e-6).all(), (t, a)
            finite_bounds = int(np.isfinite(sp.high).sum())
            assert isinstance(rew[a], (int, float)) and isinstance(term[a], bool) and isinstance(trunc[a], bool)
        assert trunc["__all__"] == (t >= 40)   # the check runs before the counter advances (mujoco_rl.py:279,288)
    assert finite_bounds > 0, "the level must declare bounded sensors"


@pytest.mark.gpu
def test_soak_keeps_every_contact():
    """Random-action rollout of the two-ant level with per-env auto-reset: the cumulative count of contacts found beyond
    an env's contact slots (mjb_buffers.ncon_dropped) stays 0, no env is reset for a non-finite state, and the state
    stays finite.  (tools/soak.py runs the same at 65536 envs x 3000 steps -> profiles/r02_soak.json.)"""
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    lv = os.path.join(os.path.dirname(os.path.abspath(__file__)), "levels")
    env = MuJoCoRL({"xmlPath": os.path.join(lv, "two_ants.xml"), "infoJson": os.path.join(lv, "info_2A.json"), "agents": ["sender", "receiver"],
                    "environmentDynamics": [P.Language], "rewardFunctions": [P.tag_distance_reward], "doneFunctions": [P.distance_done],
                    "num_envs": 2048, "maxSteps": 200, "seed": 3})
    env.reset()
    b = env.batch
    max_ncon = 0
    for t in range(600):
        obs, rew, term, trunc, _ = env.step(env.sample_actions())
        if t % 25 == 24:
            max_ncon = max(max_ncon, int(b.ncon.max()))
            done = term["__all__"] | trunc["__all__"]
            if bool(done.any()):
                env.reset(mask=done)
    assert int(b.ncon_dropped.sum()) == 0
    assert int(b.nreset.sum()) == 0
    assert 0 < max_ncon <= b.layout.maxcon
    assert bool(torch.isfinite(b.qpos).all() and torch.isfinite(b.qvel).all() and torch.isfinite(b.obs).all())


# ---- narrow phase: closed-form cases and random poses through the C-ABI (the same cases run on the kernel source under
# the host emulator and on the oracle in tests/test_collision_known_answers.py)
@pytest.mark.gpu
def test_collision_known_answers():
    from collision_cases import CASES
    from emu_harness import simple_spec
    for name, xml, qpos, ncon, dists, normal in CASES:
        model = L.Model(xml)
        spec, keep = simple_spec(model, [1], [0, 1, 5], 3, free_joint=True)
        b = _batch(model, spec, 3, keep)
        b.qpos[:, :7] = torch.tensor(qpos, dtype=torch.float32)
        b.forward(); b.sync()
        for e in range(3):
            n = int(b.ncon[e])
            assert n == ncon, (name, n, b.contact_dist[e, :n].tolist())
            assert np.allclose(sorted(b.contact_dist[e, :n].tolist()), sorted(dists), atol=2e-6), name
        assert int(b.ncon_dropped.sum()) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("which", [0, 1])
def test_random_poses_cuda_agrees_with_oracle(which):
    from emu_harness import simple_spec
    from test_collision_known_answers import RANDOM_PAIRS, random_poses
    kind, static, free = RANDOM_PAIRS[which]
    n = 1500
    model, sim, qs = random_poses(static, free, n, seed=5)
    spec, keep = simple_spec(model, [1], [0, 1, 5], 3, free_joint=True)
    b = _batch(model, spec, n, keep)
    b.qpos[:, :7] = torch.tensor(np.array(qs))
    b.forward(); b.sync()
    ncon, cd = b.ncon.cpu().numpy(), b.contact_dist.cpu().numpy()
    bad = 0
    for e, q in enumerate(qs):
        sim.qpos[:] = q.astype(np.float64)
        sim.forward()
        want = sorted(sim.contact(i)["dist"] for i in range(sim.ncon))
        got = sorted(cd[e, :ncon[e]])
        if len(want) != len(got) or (want and np.abs(np.array(want) - np.array(got)).max() > 2e-5):
            bad += 1
    # fp32 vs fp64 may flip a discrete decision on a pose that sits exactly on a feature boundary
    assert bad <= 2, (kind, bad)


@pytest.mark.gpu
@pytest.mark.parametrize("scene,n", [("ant", 1000), ("two_ants", 333)])
def test_literal_step_tile_kernel_matches_host_loop(scene, n):
    """skipFrames = 0 (the reference benchmarks' literal setting) runs the bandwidth-shaped tile kernel (lite_kernel.cuh):
    every output of 12 steps is EXACTLY the reference-order host loop's (no physics, so no rounding anywhere), for a ragged
    env count, with truncation flipping, and through the host-buffer entry point as well."""
    import os
    from common import LEVELS
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    seed, max_steps = 21, 9
    if scene == "ant":
        cfg = dict(xmlPath=os.path.join(LEVELS, "ant_rk4.xml"), agents=["torso"], rewardFunctions=[P.ant_reward_function])
        dyn, rew, done, targets, nact = [], [H.ant_reward], [], [], 3
    else:
        cfg = dict(xmlPath=os.path.join(LEVELS, "two_ants.xml"), infoJson=os.path.join(LEVELS, "info_2A.json"), agents=["sender", "receiver"],
                   environmentDynamics=[P.Language], rewardFunctions=[P.tag_distance_reward], doneFunctions=[P.distance_done])
        dyn, rew, done, targets, nact = [H.Language], [H.tag_distance_reward], [H.distance_done], ["choice_1", "choice_2"], 4
    cfg.update(freeJoint=True, skipFrames=0, maxSteps=max_steps, num_envs=n, seed=seed)
    env, env_h = MuJoCoRL(cfg), MuJoCoRL(cfg)
    agents = env.agents
    picks = [0, 1, 63, 64, 65, n // 2, n - 2, n - 1]
    mirrors = {e: _mirror_env(env, e, seed, dyn, rew, done, targets, free_joint=True, skip_frames=0, max_steps=max_steps) for e in picks}
    env.reset(); env_h.reset()
    act0 = env.batch.actions[:, :, :nact].cpu().numpy()
    for e, m in mirrors.items():
        m.reset({a: act0[e, i] for i, a in enumerate(agents)})
    hb = env_h.batch
    h_act, h_obs, h_rew, h_term, h_trunc = hb.host_arrays()
    rng = np.random.default_rng(4)
    for t in range(12):
        act = rng.uniform(-1, 1, (n, len(agents), nact)).astype(np.float32)
        if scene != "ant":
            act[:, :, 3] = rng.uniform(0, 3, (n, len(agents)))
        o, r, term, trunc, _ = env.step(torch.tensor(act))
        h_act[:, :, :nact] = act
        hb.step_host(h_act, h_obs, h_rew, h_term, h_trunc)
        b = env.batch
        for name, got in (("obs", h_obs), ("reward", h_rew), ("term", h_term), ("trunc", h_trunc)):
            assert np.array_equal(got, getattr(b, name).cpu().numpy()), (t, name)
        assert torch.equal(hb.qvel, b.qvel) and torch.equal(hb.store_i, b.store_i) and torch.equal(hb.timestep, b.timestep)
        for e, m in mirrors.items():
            mo, mr, mterm, mtrunc, _ = m.step({a: act[e, i] for i, a in enumerate(agents)})
            for i, a in enumerate(agents):
                assert np.array_equal(o[a][e].cpu().numpy().astype(np.float64), mo[a].astype(np.float32).astype(np.float64)), (t, e, a)
                assert r[a][e].item() == np.float32(mr[a]), (t, e, a)
                assert bool(trunc[a][e]) == mtrunc[a] and (not done or bool(term[a][e]) == mterm[a])
            assert bool(trunc["__all__"][e]) == mtrunc["__all__"]
        assert bool(trunc["__all__"][0]) == (t >= max_steps)
    assert int(env.batch.timestep[n - 1]) == 12


@pytest.mark.gpu
@pytest.mark.parametrize("scene,N,roll", [("2A", 65536, 320), ("1A", 65536, 80), ("S3", 16384, 320), ("3S", 16384, 320)])
def test_baseline_sizes_strided_subset_against_oracle(scene, N, roll):
    """One step from identical states AT the BASELINE env counts (C2 / C3 at 65536, C4 at 16384): the full batch runs a
    random-action rollout on the GPU (every env its own actions, so the states spread out), then 48 envs strided
    across the whole grid — every CTA position, first and last env, all copies of a packed warp — are stepped once more
    and compared with the fp64 oracle started from their (downloaded) pre-step states.  Same tolerance and exact contact-pair
    sets as test_one_step_parity."""
    model, tables, agents, fj = load_scene(scene)
    spec, keep = make_spec(model, tables, agents, fj)
    b = _batch(model, spec, N, keep)
    nq, nv, nu, ns, n_phys, A = model.nq, model.nv, model.nu, model.nsensordata, spec.n_phys_act, len(agents)
    g = torch.Generator(device="cuda"); g.manual_seed(11)
    b.reset()
    for k in range(roll):
        b.actions[:, :, :n_phys] = torch.rand((N, A, n_phys), generator=g, device="cuda") * 2 - 1
        b.physics(1)
    b.sync()
    sub = np.unique(np.concatenate([np.arange(0, N, N // 40), [1, 2, 3, N - 3, N - 2, N - 1]]))
    pre = {k: getattr(b, k)[sub].cpu().numpy().astype(np.float64) for k in ("qpos", "qvel", "warmstart", "ctrl")}
    act = (torch.rand((N, A, n_phys), generator=g, device="cuda") * 2 - 1)
    b.actions[:, :, :n_phys] = act
    act_np = act[sub].cpu().numpy().astype(np.float64)
    b.physics(1); b.sync()
    q, v, sens = b.qpos[sub].cpu().numpy(), b.qvel[sub].cpu().numpy(), b.sensordata[sub].cpu().numpy()
    ncon, cg = b.ncon[sub].cpu().numpy(), b.contact_geom[sub].cpu().numpy()
    assert len({tuple(np.round(r, 3)) for r in pre["qpos"][:, :nq]}) > len(sub) // 2, "the envs must have spread out"
    sim = OracleSim(model.blob)
    contacts = 0
    for i, e in enumerate(sub):
        sim.reset()
        sim.qpos[:] = pre["qpos"][i, :nq]; sim.qvel[:] = pre["qvel"][i, :nv]; sim.qacc_warmstart[:] = pre["warmstart"][i, :nv]
        if nu:
            sim.ctrl[:] = pre["ctrl"][i, :nu]
        for a, agent in enumerate(agents):
            idx = tables.agents_action_index[agent]
            if fj:
                sim.qvel[idx] = act_np[i, a]
            else:
                sim.ctrl[idx] = act_np[i, a]
        sim.step()
        assert rel_err(q[i, :nq], sim.qpos) < RTOL, (scene, int(e))
        assert rel_err(v[i, :nv], sim.qvel) < RTOL, (scene, int(e))
        if ns:
            assert rel_err(sens[i, :ns], sim.sensordata[:ns]) < 2e-3, (scene, int(e))
        assert sorted((int(x), int(y)) for x, y in cg[i, :ncon[i]]) == sorted(sim.contact_pairs()), (scene, int(e))
        contacts += int(ncon[i])
    assert contacts > 0
    assert int(b.ncon_dropped.sum()) == 0
