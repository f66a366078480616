"""The physics step kernel compiled at batch creation for the model's shape (csrc/spec_jit.h, DESIGN §7a): it compiles
with NVRTC for sm_100a from the sources embedded in libmjb.so, without spilling, and on the GPU it computes every buffer
bit for bit as the generic kernel does (MJB_SPEC_GENERIC) over hundreds of contact steps."""
import os
import shutil
import subprocess

import pytest

from common import LEVELS, SCENES, load_scene, make_spec
from mujoco_rl_environment_wrapper_b200 import _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SENSOR_LEVELS = os.path.join(ROOT, "tests", "sensor_levels")


def _res_usage(cubin, tmp_path):
    """(registers, stack bytes, local bytes) of the cubin's k_env, or None without cuobjdump"""
    tool = shutil.which("cuobjdump") or ("/usr/local/cuda/bin/cuobjdump" if os.path.exists("/usr/local/cuda/bin/cuobjdump") else None)
    if not tool:
        return None
    path = tmp_path / "k.cubin"
    path.write_bytes(cubin)
    out = subprocess.run([tool, "-res-usage", str(path)], capture_output=True, text=True).stdout
    line = out.split("k_env", 1)[1].splitlines()[1]
    val = {kv.split(":")[0]: int(kv.split(":")[1]) for kv in line.split() if ":" in kv and kv.split(":")[1].isdigit()}
    return val["REG"], val["STACK"], val["LOCAL"]


def _compile(model, spec, num_envs):
    try:
        return L.spec_compile(model, spec, num_envs)
    except Exception as e:   # batches then run the generic kernel (mjb_batch_spec_info); nothing to compile here
        if "libnvrtc.so.12 not found" in str(e) or "differs from the nvcc that built libmjb" in str(e):
            pytest.skip(str(e))
        raise


@pytest.mark.parametrize("scene,num_envs", [(s, 4096) for s in SCENES] + [("C1", 1)])
def test_nvrtc_compiles_every_scene_without_local_memory(scene, num_envs, tmp_path):
    model, tables, agents, fj = load_scene(scene)
    spec, keep = make_spec(model, tables, agents, fj)
    cubin, ms = _compile(model, spec, num_envs)
    assert cubin[:4] == b"\x7fELF"
    usage = _res_usage(cubin, tmp_path)
    print(f"{scene} x {num_envs}: NVRTC {ms:.0f} ms, (registers, stack, local) = {usage}")
    if usage is not None:
        reg, stack, local = usage
        assert reg <= 128 and local == 0
        # no more stack than the generic kernel (208 bytes for the unpacked C2 instantiation)
        assert stack <= 208


def test_nvrtc_shape_cache_and_value_independence():
    """models that differ only in values share one compile; another shape compiles anew"""
    model, tables, agents, fj = load_scene("2A")
    spec, keep = make_spec(model, tables, agents, fj)
    a, _ = _compile(model, spec, 4096)
    model.set_field("body_mass", model.fields["body_mass"] * 1.5)
    b, _ = L.spec_compile(model, spec, 4096)
    assert a == b
    spec2, keep2 = make_spec(model, tables, agents, fj, max_steps=7, seed=99)   # values of the spec, not its shape
    assert L.spec_compile(model, spec2, 4096)[0] == a
    spec3, keep3 = make_spec(model, tables, agents, fj, skip_frames=3)   # skip_frames is a launch argument
    assert L.spec_compile(model, spec3, 4096)[0] == a
    c1, t1, a1, f1 = load_scene("C1")
    s1, k1 = make_spec(c1, t1, a1, f1)
    assert L.spec_compile(c1, s1, 4096)[0] != a


# ---- GPU: specialised == generic, bit for bit ------------------------------------------------------------------------
def _env(cfg, generic):
    from mujoco_rl_environment_wrapper_b200 import mujoco_rl as R
    if not generic:
        return R.MuJoCoRL(dict(cfg))
    base = R.Batch

    class GenericBatch(base):
        def __init__(self, model, spec, *a, **kw):
            spec = L.EnvSpec.from_buffer_copy(spec)
            spec.flags |= L.SPEC_GENERIC
            super().__init__(model, spec, *a, **kw)

    R.Batch = GenericBatch
    try:
        return R.MuJoCoRL(dict(cfg))
    finally:
        R.Batch = base


def _buffers(env):
    import torch
    b = env.batch
    out = dict(b.buf)
    for k in ("final_obs", "params"):
        t = getattr(b, k, None)
        if isinstance(t, torch.Tensor):
            out[k] = t
    return {k: v.contiguous().view(torch.uint8) for k, v in out.items()}


def _gpu_configs():
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    two = dict(xmlPath=os.path.join(LEVELS, "two_ants.xml"), infoJson=os.path.join(LEVELS, "info_2A.json"), agents=["sender", "receiver"])
    c2 = dict(two, environmentDynamics=[P.Language], rewardFunctions=[P.tag_distance_reward], doneFunctions=[P.distance_done])
    return {
        "2A": c2,
        "C1": dict(xmlPath=os.path.join(LEVELS, "one_ant_arena.xml"), agents=["sender"]),
        "1A": dict(xmlPath=os.path.join(LEVELS, "ant_rk4.xml"), agents=["torso"], rewardFunctions=[P.ant_reward_function]),
        "3S": dict(xmlPath=os.path.join(LEVELS, "two_ants_touch_acc.xml"), agents=["sender", "receiver"], freeJoint=True, skipFrames=5),
        "imu": dict(xmlPath=os.path.join(SENSOR_LEVELS, "two_ants_imu.xml"), agents=["sender", "receiver"]),
        "autoreset-start": dict(c2, autoReset=True, maxSteps=50, startStates="pool"),
        "params-randomized": dict(c2, maxSteps=60, autoReset=True, perEnvParams=True,
                                  randomizeParams={"body_mass": [0.8, 1.2], "geom_friction": [0.5, 1.5], "actuator_gear": [0.9, 1.1],
                                                   "dof_damping": [0.5, 2.0]}),
    }


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["2A", "C1", "1A", "3S", "imu", "autoreset-start", "params-randomized"])
def test_gpu_specialised_equals_generic_bit_for_bit(name):
    import torch
    cfg = dict(_gpu_configs()[name], num_envs=4096, seed=21)
    cfg.setdefault("maxSteps", 1024)
    if cfg.get("startStates") == "pool":
        # start states: rows of a short rollout of the same scene
        warm = _env({k: v for k, v in cfg.items() if k not in ("startStates", "autoReset")}, True)
        warm.reset()
        for _ in range(20):
            warm.step(warm.sample_actions())
        n = warm.model
        cfg["startStates"] = {"qpos": warm.batch.qpos[:64, :n.nq].cpu().numpy(), "qvel": warm.batch.qvel[:64, :n.nv].cpu().numpy()}
        del warm
    spec_env, gen_env = _env(cfg, False), _env(cfg, True)
    geo = spec_env.batch.geometry()
    assert geo["specialised"], geo["spec_reason"]
    assert not gen_env.batch.geometry()["specialised"] and gen_env.batch.geometry()["spec_reason"] == "MJB_SPEC_GENERIC"
    ad = spec_env._act_dim
    g = torch.Generator(device=spec_env.device).manual_seed(3)
    for e in (spec_env, gen_env):
        e.reset()
    for k in range(400):
        act = torch.rand((4096, spec_env.batch.actions.shape[1], ad), generator=g, device=spec_env.device) * 2 - 1
        for e in (spec_env, gen_env):
            e.batch.actions[:, :, :ad].copy_(act)
            e.batch.step()
        if k == 200:   # a masked reset through the generic reset kernel on both sides
            mask = torch.arange(4096, device=spec_env.device) % 3 == 0
            for e in (spec_env, gen_env):
                e.batch.reset(mask.to(torch.uint8))
    torch.cuda.synchronize()
    a, b = _buffers(spec_env), _buffers(gen_env)
    assert sorted(a) == sorted(b)
    diff = [k for k in a if not torch.equal(a[k], b[k])]
    assert not diff, diff
