"""Single-agent adapters over the batched environment (SURVEY 8f row 2).

Same constructor / step / reset contract as MuJoCo_Gym/wrappers.py:12-142.  With `num_envs > 1` every
returned value keeps its leading `num_envs` dimension (a vector-env view).  Two stale spots of the
reference are repaired rather than reproduced: `GymWrapper` reads the spaces through the methods
(`wrappers.py:110-111` treats them as attributes) and tolerates a missing `terminations["__all__"]`
(present only when done functions are configured, `mujoco_rl.py:281-286`)."""
import torch


class GymnasiumWrapper:
    metadata = {"render_modes": ["human", "none"], "render_fps": 4}

    def __init__(self, environment, agent: str, render_mode="none"):
        self.environment, self.agent, self.render_mode = environment, agent, render_mode
        if len(self.environment.agents) > 1:
            raise Exception("Environment has too many agents. Only one agent is allowed in a gym environment.")
        self.observation_space = environment.observation_space(agent)
        self.action_space = environment.action_space(agent)

    def step(self, action):
        """With the environment's `autoReset`, `info` carries `final_observation` (the last observation of an episode the
        step ended, the returned one being the next episode's first) and its mask `_final_observation`."""
        observations, rewards, terminations, truncations, infos = self.environment.step({self.agent: action})
        return observations[self.agent], rewards[self.agent], terminations[self.agent], truncations["__all__"], infos[self.agent]

    def reset(self, *, seed=1, options=None):
        """`options`: passed to the environment's reset, e.g. {"qpos": ..., "qvel": ...} to start from a given state."""
        observations, infos = self.environment.reset(options=options)
        return observations[self.agent], infos

    def render(self):
        pass


class GymWrapper(GymnasiumWrapper):
    def step(self, action):
        observations, rewards, terminations, truncations, infos = self.environment.step({self.agent: action})
        term_all = terminations.get("__all__", terminations[self.agent])
        trunc_all = truncations["__all__"]
        done = (term_all | trunc_all) if torch.is_tensor(term_all) else bool(term_all or trunc_all)
        return observations[self.agent], rewards[self.agent], done, infos[self.agent]

    def reset(self):
        observations, infos = self.environment.reset()
        return observations[self.agent]
