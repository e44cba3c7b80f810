"""OctoCrawl-v0 on the B200 kernel.

Host-side mirror of `/root/reference/gym_softrobot/envs/octopus/crawl_env.py` (`CrawlEnv`, lines 34-313) and
`build_octopus_muscles` (`envs/octopus/build_muscle_octopus.py:70-179`): eight tapered arms (radius 13 mm -> 4.2 mm)
at 22.5 + 45 i degrees around a light rigid head, `FixedJoint2Rigid` joints, `BodyBoundaryCondition` on the head, an
`AnalyticalLinearDamper` per arm, one `ControllableFixConstraint` ("sucker") per arm, and COOMM's `ApplyMuscles` of
which only the transverse muscle is activated.  Per arm the action is (sucker location, activation, reduction ratio).
The substep loop (crawl_env.py:253-254) is one `sr_step` launch.

COOMM is a third-party package outside the reference tree: its published muscle model is restated (DESIGN.md 2).
"""
from typing import Optional

import numpy as np

from .. import _native as nat
from .fork import ForkableVectorEnv
from ..compat import Box, Env
from .soft_pendulum import _advance_time

_ARM = dict(base_length=0.25, base_radius=0.013, tip_radius=0.0042, density=1000.0, youngs_modulus=1.5e4,
            shear_modulus=1.5e4 / (1.0 + 0.5))
_HEAD_RADIUS, _HEAD_DENSITY = 0.04, 50.0
_JOINT = dict(k=1e6, kt=1e2, nu=1e-3)
_DAMPER_TIME_STEP = 7e-5      # the literal the build passes to AnalyticalLinearDamper (build_muscle_octopus.py:102-107)
_N_ARM = 8


def crawl_init_params(n_arm=_N_ARM):
    """[9 * (n_arm + 1)] start / direction / normal of every arm, then of the head cylinder
    (build_muscle_octopus.py:88-118)."""
    angles = [45.0 / 2 + 45.0 * i for i in range(n_arm)]
    row = []
    for ang in angles:
        c, s = np.cos(np.deg2rad(ang)), np.sin(np.deg2rad(ang))
        row += [c * _HEAD_RADIUS, s * _HEAD_RADIUS, 0.0, c, s, 0.0, 0.0, 0.0, 1.0]
    row += [0.0, 0.0, -_ARM["base_radius"] * 2, 0.0, 0.0, 1.0, 0.0, 1.0, 0.0]
    return np.array([row]), angles


class OctoCrawlVectorEnv(ForkableVectorEnv):
    """N independent OctoCrawl-v0 envs (torch CUDA I/O), one physics launch per env-step; actions float [n_env, 24]."""

    PER_ENV = ("step_count", "prev_action", "_final")   # per-env host state (copy_envs)

    def __init__(self, n_env, final_time=10.0, time_step=5.0e-5, recording_fps=25, n_elems=20,
                 config_random_final_time=False, device: int = 0, autoreset: bool = True):
        import torch
        self.torch = torch
        self.n_env, self.n_arm, self.n_elems, self.n_seg, self.n_action = n_env, _N_ARM, n_elems, n_elems - 1, 3
        self.final_time, self.time_step = final_time, time_step
        self.step_skip = int(1.0 / (recording_fps * time_step))
        self.config_random_final_time = config_random_final_time
        self.device = torch.device(f"cuda:{device}")
        self.autoreset = autoreset
        self.shared_space = 17
        obs_dim = self.n_arm * (self.n_seg + (n_elems + 1) * 4 + self.n_action + self.n_arm + self.shared_space)
        self.single_action_space = Box(0.0, 1.0, shape=(self.n_arm * self.n_action,), dtype=np.float32)
        self.single_observation_space = Box(-np.inf, np.inf, shape=(obs_dim,), dtype=np.float32)
        self._init, angles = crawl_init_params(self.n_arm)
        # the damper's coefficients are exp(-nu * 7e-5 ...) whatever the env's time step: same exponent through nu' = nu 7e-5 / dt
        damp = 0.20 * 1e-2 * (_DAMPER_TIME_STEP / time_step)
        self.handle = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n_elems, dt=time_step, gravity=(0.0, 0.0, 0.0),
                                 damping_constant=damp, bc_kind=nat.BC_FREE, device=device, n_rod=self.n_arm,
                                 head=dict(length=_ARM["base_radius"] * 2, radius=_HEAD_RADIUS, density=_HEAD_DENSITY),
                                 joint=dict(radius=_HEAD_RADIUS, angles_deg=angles, **_JOINT), sucker_index=0,
                                 tm_muscle=dict(max_stress=1.0, radius_ref=_ARM["base_radius"]), **_ARM)
        self._scratch = (torch.empty((n_env, 6), dtype=torch.float32, device=self.device),
                         torch.empty(n_env, dtype=torch.float64, device=self.device),
                         torch.empty(n_env, dtype=torch.uint8, device=self.device))
        self._target = torch.tensor([5.0, 0.0], dtype=torch.float32, device=self.device)
        self._eye = torch.eye(self.n_arm, dtype=torch.float64, device=self.device)
        n_max = int(10.0 / (self.step_skip * time_step)) + int(final_time / (self.step_skip * time_step)) + 8
        table, t = [np.float64(0.0)], np.float64(0.0)
        for _ in range(n_max):
            t = _advance_time(t, time_step, self.step_skip)
            table.append(t)
        self._time_table = torch.as_tensor(np.array(table), device=self.device)
        self._final = torch.full((n_env,), float(final_time), dtype=torch.float64, device=self.device)
        self._rng = np.random.default_rng()
        self.step_count = torch.zeros(n_env, dtype=torch.int64, device=self.device)
        # (set at construction and by set_action only, like the reference: crawl_env.py:108-110,246)
        self.prev_action = torch.zeros((n_env, self.n_arm, self.n_action), dtype=torch.float32, device=self.device)

    # -- helpers -----------------------------------------------------------------------------
    def _head_xy(self):
        return self.handle.head_tensor()[:, 0:2]

    def _obs(self):
        torch = self.torch
        f = self.handle.fields()
        N, A = self.n_env, self.n_arm
        sh = lambda t: t.reshape((N, A) + tuple(t.shape[-2:]))
        kappa = sh(f["kappa"])[:, :, 0, :]
        x, v = sh(f["position_collection"]), sh(f["velocity_collection"])
        hd = self.handle.head_tensor()
        # get_shared_state: target, head position, head velocity, director_collection[:, :, 0].ravel() — cast to float32
        shared = torch.cat([self._target.expand(N, 2).double(), hd[:, 0:3], hd[:, 3:6], hd[:, 6:15]], dim=1).float().double()
        obs = torch.cat([kappa, x[:, :, 0, :], x[:, :, 1, :], v[:, :, 0, :], v[:, :, 1, :], self.prev_action.double(),
                         self._eye.expand(N, A, A), shared[:, None, :].expand(N, A, self.shared_space)], dim=2)
        return torch.nan_to_num(obs.float().reshape(N, -1))

    def _reset_envs(self, idx=None):
        torch = self.torch
        n = self.n_env if idx is None else int(idx.numel())
        init = torch.as_tensor(np.repeat(self._init, n, axis=0), device=self.device).contiguous()
        self.handle.reset(init, None if idx is None else idx.to(torch.int32).contiguous())
        A = self.n_arm
        view = lambda t: t.unflatten(0, (self.n_env, A))
        sel = slice(None) if idx is None else idx
        # a fresh build: SuckerController(index=0) (reduction_ratio 1.0) turned on, muscles at rest
        view(self.handle.sucker_tensor())[sel] = 1.0
        view(self.handle.sucker_index_tensor())[sel] = 0
        view(self.handle.tm_activation_tensor())[sel] = 0.0
        if self.config_random_final_time:
            self._final[sel] = torch.as_tensor(self._rng.uniform(3.0, 10.0, size=n), device=self.device)

    def reset(self, seed: Optional[int] = None):
        if seed is not None:
            self._rng = np.random.default_rng(seed)
        self._reset_envs()
        self.step_count.zero_()
        return self._obs(), {}

    def set_final_time(self, final_time):
        self._final[:] = torch_as(self.torch, final_time, self.device)

    def set_action(self, action):
        torch = self.torch
        a = action.to(device=self.device, dtype=torch.float32).reshape(self.n_env, self.n_arm, self.n_action)
        # crawl_env.py:236-243: index = int(np.clip(location * n_elems, 0, n_elems - 1)) on the float32 action
        self.handle.sucker_index_tensor()[:] = torch.clamp(a[:, :, 0] * self.n_elems, 0, self.n_elems - 1).to(torch.int32).reshape(-1)
        self.handle.tm_activation_tensor()[:] = a[:, :, 1].double().reshape(-1)
        self.handle.sucker_tensor()[:] = a[:, :, 2].double().reshape(-1)
        self.prev_action = a.clone()

    def step(self, action):
        torch = self.torch
        self.set_action(action)
        target = self._target.double()
        before = self._head_xy().clone()
        obs6, rew, term = self._scratch
        self.handle.step(None, self.step_skip, obs6, rew, term)
        self.step_count += 1
        obs = self._obs()
        invalid = term.bool()        # NaN in any arm's position / velocity
        after = self._head_xy()
        d_after = (target - after).norm(dim=1)
        forward = ((target - before).norm(dim=1) - d_after) * 1e2
        reached = (d_after < 0.2) & ~invalid
        reward = torch.where(invalid, torch.full_like(forward, -5.0), forward + torch.where(reached, 5.0, 0.0))
        terminated = invalid | reached
        time = self._time_table[self.step_count.clamp(max=self._time_table.numel() - 1)]
        truncated = ~terminated & (time > self._final)
        bad = torch.isnan(reward)
        terminated = terminated | bad
        # `reward -= 5; reward = min(self.reward_range, reward)`: python's min(100.0, nan) is 100.0
        reward = torch.where(bad, torch.full_like(reward, 100.0), torch.clamp(reward, max=100.0))
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


def torch_as(torch, value, device):
    return torch.as_tensor(value, dtype=torch.float64, device=device)


class CrawlEnv(Env):
    """Drop-in for the reference `CrawlEnv` (same kwargs; crawl_env.py:58-66): a batch of one."""

    metadata = {"render_modes": ["rgb_array"], "render_fps": 25, "multiagent": ["PyMARL"]}

    def __init__(self, final_time=10.0, time_step=5.0e-5, recording_fps=25, n_elems=20,
                 config_random_final_time=False, render_mode: Optional[str] = None, device: int = 0):
        super().__init__()
        if render_mode not in {None, *self.metadata["render_modes"]}:
            raise ValueError(f"Unsupported render mode: {render_mode}")
        self.render_mode = render_mode
        self._vec = OctoCrawlVectorEnv(1, final_time, time_step, recording_fps, n_elems, False, device, autoreset=False)
        self.final_time, self.time_step, self.recording_fps = final_time, time_step, recording_fps
        self.step_skip = self._vec.step_skip
        self.n_arm = self.n_agent = _N_ARM
        self.n_elems, self.n_seg, self.n_action = n_elems, n_elems - 1, 3
        self.shared_space, self.grid_size, self.reward_range = 17, 1, 100.0
        self.action_space = self._vec.single_action_space
        self.observation_space = self._vec.single_observation_space
        self.config_random_final_time = config_random_final_time
        self.time = np.float64(0.0)
        self.counter = 0

    @property
    def agent_id(self):
        return ["LF1", "LF2", "LB2", "LB1", "RB1", "RB2", "RF2", "RF1"]

    def get_env_info(self):
        return dict(n_actions=self.n_action, n_agents=8)

    def reset(self, *, seed: Optional[int] = None, options: Optional[dict] = None):
        super().reset(seed=seed)
        if self.config_random_final_time:
            self.final_time = self.np_random.uniform(3.0, 10.0)
        self._vec.set_final_time(float(self.final_time))
        obs, _ = self._vec.reset()
        self.time = np.float64(0.0)
        self.counter = 0
        self._target = np.array([5, 0], dtype=np.float32)
        return obs[0].cpu().numpy(), {}

    def step(self, action):
        import torch
        a = torch.as_tensor(np.asarray(action, dtype=np.float32).reshape(1, -1), device=self._vec.device)
        obs, reward, term, trunc, _ = self._vec.step(a)
        self.time = _advance_time(self.time, self.time_step, self.step_skip)
        terminated = bool(term[0])
        truncated = (not terminated) and bool(self.time > self.final_time)
        self.counter += 1
        return obs[0].cpu().numpy(), float(reward[0].item()), terminated, truncated, {"time": self.time}

    def arm_states(self):
        return {k: v[0].cpu().numpy() for k, v in self._vec.fields().items()}

    def head_state(self):
        return self._vec.handle.head_tensor()[0].cpu().numpy()

    def render(self):
        return None

    def close(self):
        self._vec.close()
