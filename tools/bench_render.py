"""Agent-camera raycaster throughput (SURVEY 8 f4) -> gpurun_out/r01_render.json.
C2 scene with the reference's two agent cameras, 64x64 (the reference's default sensorResolution), settled
state; the output tensor (N x 2 x 64 x 64 x 3 bytes) is larger than L2 from N = 5200 up.
Columns (CUDA events, L2 not flushed): `ms_per_render` colour only (mjb_render); `ms_rgb_depth_seg` all three channels
(mjb_render_ex); `ms_masked` colour, depth and segmentation of ceil(N / 1025) envs picked by a mask (the share of envs an
auto-reset step with staggered episodes of 1024 steps ends, whose last frames render_ex(final=True) draws)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL  # noqa: E402

LV = os.path.join(ROOT, "tests", "levels")
res = []
for n, wh in ((4096, 64), (16384, 64), (4096, 128)):
    env = MuJoCoRL({"xmlPath": os.path.join(LV, "two_ants_cams.xml"), "agents": ["sender", "receiver"], "agentCameras": True,
                    "num_envs": n, "sensorResolution": (wh, wh)})
    env.reset()
    for _ in range(150):
        env.step(env.sample_actions())
    b = env.batch
    out = b.render([0, 1], wh, wh)
    for _ in range(3):
        b.render([0, 1], wh, wh, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 20

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps
    ms = timed(lambda: b.render([0, 1], wh, wh, out=out))
    full = b.render_ex([0, 1], wh, wh, depth=True, segmentation=True)
    ms_all = timed(lambda: b.render_ex([0, 1], wh, wh, depth=True, segmentation=True, out=full))
    mask = torch.zeros(n, dtype=torch.bool, device=b.device)
    n_masked = -(-n // 1025)
    mask[torch.randperm(n, generator=torch.Generator().manual_seed(0))[:n_masked].to(b.device)] = True
    ms_masked = timed(lambda: b.render_ex([0, 1], wh, wh, depth=True, segmentation=True, mask=mask, out=full))
    rays = n * 2 * wh * wh
    r = {"envs": n, "cameras": 2, "resolution": [wh, wh], "ms_per_render": ms, "ms_rgb_depth_seg": ms_all,
         "ms_masked": ms_masked, "masked_envs": n_masked, "frames_per_s": n * 2 / (ms * 1e-3),
         "rays_per_s": rays / (ms * 1e-3), "ray_geom_tests_per_s": rays * env.model.ngeom / (ms * 1e-3),
         "output_GBps": out.numel() / (ms * 1e-3) / 1e9, "lit_fraction": float((out.view(-1, 3).sum(1) > 0).float().mean())}
    print(json.dumps(r), flush=True)
    res.append(r)
    del env, b, out, full
    torch.cuda.empty_cache()
os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
json.dump(res, open(os.path.join(ROOT, "gpurun_out", "r01_render.json"), "w"), indent=1)
