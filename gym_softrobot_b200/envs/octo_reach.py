"""OctoReach-v0 on the B200 kernel.

Host-side mirror of `/root/reference/gym_softrobot/envs/octopus/reach_env.py` (`ReachEnv`, lines 36-302) over
`build_octopus_muscles` (`envs/octopus/build_muscle_octopus.py:70-179`): eight tapered arms around a rigid head that
`OneEndFixedBC` pins (reach_env.py:128-132), and COOMM's `ApplyMuscles` with ALL THREE muscle layers of
`create_es_muscle_layers` (envs/octopus/build.py:292-338) driven by per-element activations: the action is
[8 arms x 3 muscles x n_elems] in [0, 1] (reach_env.py:214-227).  The reward is the squared distance of the closest arm
tip to a random target.  The substep loop (reach_env.py:233-234) is one `sr_step` launch of the muscle-layer kernel.

COOMM is a third-party package outside the reference tree: its published muscle model is restated (DESIGN.md 2).
"""
from typing import Optional

import numpy as np

from .. import _native as nat
from .fork import ForkableVectorEnv
from ..compat import Box, Env
from .octo_crawl import _ARM, _DAMPER_TIME_STEP, _HEAD_DENSITY, _HEAD_RADIUS, _JOINT, _N_ARM, crawl_init_params
from .soft_pendulum import _advance_time

_N_MUSCLE = 3
_LM_MAX_STRESS, _TM_MAX_STRESS = 0.5, 1.0


def es_longitudinal_positions():
    """ratio_muscle_position (0, -6/9, 0) rotated by muscle_init_angle = +-pi/2 about the arm axis (build.py:303-328)."""
    out = []
    for ang in (np.pi / 2, -np.pi / 2):
        c, s = np.cos(ang), np.sin(ang)
        out.append((c * 0.0 - s * (-6 / 9), s * 0.0 + c * (-6 / 9)))
    return out


class OctoReachVectorEnv(ForkableVectorEnv):
    """N independent OctoReach-v0 envs (torch CUDA I/O), one physics launch per env-step; actions float
    [n_env, 8 * 3 * n_elems]."""

    PER_ENV = ("step_count", "prev_action", "target")   # per-env host state (copy_envs)

    def __init__(self, n_env, final_time=5.0, time_step=5.0e-5, recording_fps=25, n_elems=20, device: int = 0,
                 autoreset: bool = True):
        import torch
        self.torch = torch
        self.n_env, self.n_arm, self.n_elems, self.n_seg = n_env, _N_ARM, n_elems, n_elems - 1
        self.n_muscle, self.n_action = _N_MUSCLE, n_elems * _N_MUSCLE
        self.final_time, self.time_step = final_time, time_step
        self.step_skip = int(1.0 / (recording_fps * time_step))
        self.device = torch.device(f"cuda:{device}")
        self.autoreset = autoreset
        self.shared_space = 18
        obs_dim = self.n_arm * (self.n_seg + (n_elems + 1) * 4 + self.n_action + self.n_arm + self.shared_space)
        self.single_action_space = Box(0.0, 1.0, shape=(self.n_arm * self.n_action,), dtype=np.float32)
        self.single_observation_space = Box(-np.inf, np.inf, shape=(obs_dim,), dtype=np.float32)
        self._init, angles = crawl_init_params(self.n_arm)
        damp = 0.20 * 1e-2 * (_DAMPER_TIME_STEP / time_step)     # (see octo_crawl.py: the damper's literal time step)
        self.handle = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n_elems, dt=time_step, gravity=(0.0, 0.0, 0.0),
                                 damping_constant=damp, bc_kind=nat.BC_FREE, device=device, n_rod=self.n_arm,
                                 head=dict(length=_ARM["base_radius"] * 2, radius=_HEAD_RADIUS, density=_HEAD_DENSITY),
                                 joint=dict(radius=_HEAD_RADIUS, angles_deg=angles, **_JOINT),
                                 tm_muscle=dict(max_stress=_TM_MAX_STRESS, radius_ref=_ARM["base_radius"]),
                                 muscle_layers=dict(lm_max_stress=_LM_MAX_STRESS, lm_positions=es_longitudinal_positions()),
                                 head_fixed=True, **_ARM)
        self._scratch = (torch.empty((n_env, 6), dtype=torch.float32, device=self.device),
                         torch.empty(n_env, dtype=torch.float64, device=self.device),
                         torch.empty(n_env, dtype=torch.uint8, device=self.device))
        self._eye = torch.eye(self.n_arm, dtype=torch.float64, device=self.device)
        n_max = int(final_time / (self.step_skip * time_step)) + 8
        table, t = [np.float64(0.0)], np.float64(0.0)
        for _ in range(n_max):
            t = _advance_time(t, time_step, self.step_skip)
            table.append(t)
        self._time_table = torch.as_tensor(np.array(table), device=self.device)
        self._rng = np.random.default_rng()
        self.step_count = torch.zeros(n_env, dtype=torch.int64, device=self.device)
        self.target = torch.zeros((n_env, 3), dtype=torch.float64, device=self.device)
        # (set at construction and by set_action only, like the reference: reach_env.py:97-99,228)
        self.prev_action = torch.zeros((n_env, self.n_arm, self.n_action), dtype=torch.float32, device=self.device)

    # -- helpers -----------------------------------------------------------------------------
    def _obs(self):
        torch = self.torch
        f = self.handle.fields()
        N, A = self.n_env, self.n_arm
        kappa = f["kappa"][:, :, 0, :]
        x, v = f["position_collection"], f["velocity_collection"]
        hd = self.handle.head_tensor()
        # shared state: target, head position, head velocity, director_collection[:, :, 0].ravel() — cast to float32
        shared = torch.cat([self.target, hd[:, 0:3], hd[:, 3:6], hd[:, 6:15]], dim=1).float().double()
        obs = torch.cat([kappa, x[:, :, 0, :], x[:, :, 1, :], v[:, :, 0, :], v[:, :, 1, :], self.prev_action.double(),
                         self._eye.expand(N, A, A), shared[:, None, :].expand(N, A, self.shared_space)], dim=2)
        return torch.nan_to_num(obs.float().reshape(N, -1))

    def _reset_envs(self, idx=None, target=None):
        torch = self.torch
        n = self.n_env if idx is None else int(idx.numel())
        init = torch.as_tensor(np.repeat(self._init, n, axis=0), device=self.device).contiguous()
        self.handle.reset(init, None if idx is None else idx.to(torch.int32).contiguous())
        sel = slice(None) if idx is None else idx
        act = self.handle.muscle_activation_tensor().unflatten(0, (self.n_env, self.n_arm))
        act[sel] = 0.0                                           # a fresh build: muscles at rest
        if target is None:    # self.np_random.random(3) * sum(rest_lengths)  (reach_env.py:166-168)
            target = self._rng.random((n, 3)) * _ARM["base_length"]
        self.target[sel] = torch.as_tensor(np.asarray(target, dtype=np.float64).reshape(n, 3), device=self.device)

    def reset(self, seed: Optional[int] = None, target=None):
        if seed is not None:
            self._rng = np.random.default_rng(seed)
        self._reset_envs(None, target)
        self.step_count.zero_()
        return self._obs(), {}

    def set_action(self, action):
        torch = self.torch
        a = action.to(device=self.device, dtype=torch.float32).reshape(self.n_env, self.n_arm, self.n_action)
        # reach_env.py:219-225: muscle j of arm i takes action[i, n_elems * j : n_elems * (j + 1)]
        self.handle.muscle_activation_tensor()[:] = a.double().reshape(self.n_env * self.n_arm, self.n_muscle, self.n_elems)
        self.prev_action = a.clone()

    def step(self, action):
        torch = self.torch
        self.set_action(action)
        obs6, rew, term = self._scratch
        self.handle.step(None, self.step_skip, obs6, rew, term)
        self.step_count += 1
        obs = self._obs()
        invalid = term.bool()        # NaN in any arm's position / velocity
        tips = self.handle.fields()["position_collection"][:, :, :, -1]          # [N, 8, 3]
        dist = (self.target[:, None, :] - tips).norm(dim=2)
        dmin = dist.min(dim=1).values / 0.25
        forward = -(dmin ** 2)
        reached = (dmin < 0.1) & ~invalid
        reward = torch.where(invalid, torch.full_like(forward, -5.0), forward + torch.where(reached, 5.0, 0.0))
        terminated = invalid | reached
        time = self._time_table[self.step_count.clamp(max=self._time_table.numel() - 1)]
        truncated = ~invalid & (time > self.final_time)           # (the reference sets it whether or not the tip arrived)
        bad = torch.isnan(reward)
        terminated = terminated | bad
        reward = torch.where(bad, torch.full_like(reward, -5.0), torch.clamp(reward, max=100.0))
        info = {"time": time}
        done = terminated | truncated
        if self.autoreset and bool(done.any()):
            idx = torch.nonzero(done).flatten()
            info["final_obs"], info["reset_idx"] = obs[idx].clone(), idx
            self._reset_envs(idx)
            self.step_count[idx] = 0
            obs[idx] = self._obs()[idx]
        return obs, reward, terminated, truncated, info

    def fields(self):
        return self.handle.fields()

    def close(self):
        self.handle.close()


class ReachEnv(Env):
    """Drop-in for the reference `ReachEnv` (same kwargs; reach_env.py:50-57): a batch of one."""

    metadata = {"render_modes": ["rgb_array"], "render_fps": 25}

    def __init__(self, final_time=5.0, time_step=5.0e-5, recording_fps=25, n_elems=20,
                 render_mode: Optional[str] = None, device: int = 0):
        super().__init__()
        if render_mode not in {None, *self.metadata["render_modes"]}:
            raise ValueError(f"Unsupported render mode: {render_mode}")
        self.render_mode = render_mode
        self._vec = OctoReachVectorEnv(1, final_time, time_step, recording_fps, n_elems, device, autoreset=False)
        self.final_time, self.time_step, self.recording_fps = final_time, time_step, recording_fps
        self.total_steps = int(final_time / time_step)
        self.step_skip = self._vec.step_skip
        self.n_arm, self.n_muscle = _N_ARM, _N_MUSCLE
        self.n_elems, self.n_seg, self.n_action = n_elems, n_elems - 1, n_elems * _N_MUSCLE
        self.grid_size, self.reward_range = 1, 100.0
        self.action_space = self._vec.single_action_space
        self.observation_space = self._vec.single_observation_space
        self.time = np.float64(0.0)
        self.counter = 0
        self._target = np.zeros(3)

    def get_env_info(self):
        return dict(n_actions=self.n_action, n_agents=8)

    def reset(self, *, seed: Optional[int] = None, options: Optional[dict] = None):
        super().reset(seed=seed)
        # sum(rest_lengths) of arm 0 as straight_rod lays it out (norms of the differences of the linspace positions)
        ang = np.deg2rad(45.0 / 2)
        d = np.array([np.cos(ang), np.sin(ang), 0.0])
        pos = (d * _HEAD_RADIUS)[:, None] + d[:, None] * np.linspace(0.0, _ARM["base_length"], self.n_elems + 1)[None, :]
        rest = np.linalg.norm(pos[:, 1:] - pos[:, :-1], axis=0)
        self._target = self.np_random.random(3) * sum(rest)
        obs, _ = self._vec.reset(target=self._target[None, :])
        self.time = np.float64(0.0)
        self.counter = 0
        return obs[0].cpu().numpy(), {}

    def step(self, action):
        import torch
        a = torch.as_tensor(np.asarray(action, dtype=np.float32).reshape(1, -1), device=self._vec.device)
        obs, reward, term, trunc, _ = self._vec.step(a)
        self.time = _advance_time(self.time, self.time_step, self.step_skip)
        terminated = bool(term[0])
        invalid = terminated and float(reward[0].item()) == -5.0
        truncated = (not invalid) and bool(self.time > self.final_time)
        self.counter += 1
        return obs[0].cpu().numpy(), float(reward[0].item()), terminated, truncated, {"time": self.time}

    def compute_reward(self, achieved_goal, desired_goal, _info=None):
        eps = 0.01
        dist = np.linalg.norm(np.asarray(achieved_goal) - np.asarray(desired_goal), axis=-1)
        return -(dist > eps).astype(np.float32)

    def arm_states(self):
        return {k: v[0].cpu().numpy() for k, v in self._vec.fields().items()}

    def head_state(self):
        return self._vec.handle.head_tensor()[0].cpu().numpy()

    def render(self):
        return None

    def close(self):
        self._vec.close()
