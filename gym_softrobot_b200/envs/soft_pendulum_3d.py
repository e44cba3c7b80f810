"""SoftPendulum3D-v0 on the B200 kernel.

Host-side mirror of `/root/reference/gym_softrobot/envs/soft_pendulum_3d/soft_pendulum_3d.py`
(`SoftPendulum3DEnv`, lines 20-158) and `.../soft_pendulum_3d/build.py:43-86`: a vertical rod on a
commanded moving base, gravity, `AnalyticalLinearDamper(1.0)` + `LaplaceDissipationFilter(7)`.
The base-controller update of `set_action` (lines 106-120), the substep loop (line 126-127), the tilt
angle, reward and observation are all evaluated inside the one `sr_step` launch.

`n_elems` may be up to 4095: rods of more than 1023 elements run one per thread-block cluster.  A finer rod
needs a correspondingly smaller `time_step` (the stable step shrinks with the element length: the default 1e-4
suits 50 elements; 2048 elements are stepped with 1e-6, e.g. `n_elems=2048, time_step=1e-6, recording_fps=2500`).
"""
from typing import Optional

import numpy as np

from .. import _native as nat
from .fork import ForkableVectorEnv
from ..compat import Box, Env
from .soft_pendulum import _advance_time

_ROD = dict(base_length=1.0, base_radius=0.1, density=4000.0, youngs_modulus=1e6)  # build.py:55-64
_GRAVITY = (0.0, 0.0, -9.80665)
_BASE_STEP, _BASE_LIMIT = 1e-3, 0.5   # soft_pendulum_3d.py:55-56


def pendulum3d_init_params(tilt_deg):
    """start / direction / normal rows for `sr_reset` (build.py:51-53); tilt_deg ~ U(-1, 1)."""
    tilt = np.deg2rad(np.atleast_1d(np.asarray(tilt_deg, dtype=np.float64)))
    init = np.zeros((tilt.shape[0], 9))
    init[:, 3] = np.sin(tilt)
    init[:, 5] = np.cos(tilt)
    init[:, 7] = 1.0
    return init


def _make_handle(n_env, n_elems, time_step, step_skip, device):
    return nat.Handle(
        model=nat.MODEL_SOFT_PENDULUM_3D, n_env=n_env, n_elem=n_elems, dt=time_step, gravity=_GRAVITY,
        damping_constant=1.0, laplace_filter_order=7, bc_kind=nat.BC_MOVING_BASE,
        damping_before_constraints=False, device=device, base_step=_BASE_STEP, base_limit=_BASE_LIMIT,
        base_move_period=step_skip * time_step, **_ROD,
    )


class SoftPendulum3DEnv(Env):
    """Drop-in for the reference `SoftPendulum3DEnv` (same kwargs; soft_pendulum_3d.py:25-33)."""

    metadata = {"render_modes": ["rgb_array"], "render_fps": 25}

    def __init__(self, final_time: float = 5.0, time_step: float = 1.0e-4, recording_fps: int = 25,
                 n_elems: int = 50, config_generate_video: bool = False,
                 render_mode: Optional[str] = None, device: int = 0):
        super().__init__()
        if render_mode not in {None, *self.metadata["render_modes"]}:
            raise ValueError(f"Unsupported render mode: {render_mode}")
        self.render_mode = render_mode
        self.final_time, self.time_step, self.recording_fps = final_time, time_step, recording_fps
        self.total_steps = int(final_time / time_step)
        self.step_skip = int(1.0 / (recording_fps * time_step))
        self.n_elems, self.n_seg, self.n_action = n_elems, n_elems - 1, 2
        self.action_space = Box(low=-1.0, high=1.0, shape=(2,), dtype=np.float32)
        self.observation_space = Box(low=-np.inf, high=np.inf, shape=(9,), dtype=np.float32)
        self._prev_action = np.zeros(2, dtype=np.float32)
        self.base_step, self.base_limit = _BASE_STEP, _BASE_LIMIT
        self.config_generate_video = config_generate_video
        self._device = device
        self._handle = None
        self.time = np.float64(0.0)
        self.counter = 0

    def reset(self, *, seed: Optional[int] = None, options: Optional[dict] = None):
        Env.reset(self, seed=seed)
        if self._handle is None:
            self._handle = _make_handle(1, self.n_elems, self.time_step, self.step_skip, self._device)
        self._prev_action.fill(0.0)
        self._handle.reset_host(pendulum3d_init_params(self.np_random.uniform(-1.0, 1.0)))
        self.time = np.float64(0.0)
        self.counter = 0
        return self.get_state(), {}

    def get_state(self):
        import torch
        dev = f"cuda:{self._device}"
        obs = torch.empty((1, 9), dtype=torch.float32, device=dev)
        pa = torch.as_tensor(self._prev_action, device=dev).reshape(1, 2).contiguous()
        self._handle.observe(pa, obs)
        return obs.cpu().numpy()[0]

    def step(self, action):
        if not self.action_space.contains(action):
            raise ValueError(f"Action {action!r} is outside {self.action_space}")
        a = np.asarray(action, dtype=np.float32).reshape(2)
        self._prev_action[:] = a
        obs, reward, terminated = self._handle.step_host(a.reshape(1, 2), self.step_skip)
        self.time = _advance_time(self.time, self.time_step, self.step_skip)
        tilt = float(self._handle.aux_tensor()[0, 6].item())
        self.counter += 1
        return (obs[0].copy(), float(reward[0]), bool(terminated[0]), bool(self.time >= self.final_time),
                {"time": self.time, "tilt": tilt})

    def rod_state(self):
        return {k: v[0].cpu().numpy() for k, v in self._handle.fields().items()}

    def render(self):
        return None

    def close(self):
        if self._handle is not None:
            self._handle.close()
            self._handle = None


class SoftPendulum3DVectorEnv(ForkableVectorEnv):
    """N independent SoftPendulum3D-v0 envs, one kernel launch per env-step (torch CUDA I/O)."""

    PER_ENV = ("step_count",)   # per-env host state (copy_envs)

    def __init__(self, n_env, final_time=5.0, time_step=1.0e-4, recording_fps=25, n_elems=50,
                 device: int = 0, autoreset: bool = True, env_offset: int = 0):
        import torch
        self.torch = torch
        self.n_env, self.n_elems = n_env, n_elems
        self.final_time, self.time_step = final_time, time_step
        self.step_skip = int(1.0 / (recording_fps * time_step))
        self.device = torch.device(f"cuda:{device}")
        self.env_offset, self.autoreset = env_offset, autoreset
        self.single_action_space = Box(low=-1.0, high=1.0, shape=(2,), dtype=np.float32)
        self.single_observation_space = Box(low=-np.inf, high=np.inf, shape=(9,), dtype=np.float32)
        self.handle = _make_handle(n_env, n_elems, time_step, self.step_skip, device)
        self.obs = torch.empty((n_env, 9), dtype=torch.float32, device=self.device)
        self.reward = torch.empty(n_env, dtype=torch.float64, device=self.device)
        self.terminated = torch.empty(n_env, dtype=torch.uint8, device=self.device)
        n_max = int(final_time / (self.step_skip * time_step)) + 8
        table, t = [np.float64(0.0)], np.float64(0.0)
        for _ in range(n_max):
            t = _advance_time(t, time_step, self.step_skip)
            table.append(t)
        self._time_table = np.array(table)
        self._first_truncated = int(np.argmax(self._time_table >= final_time))   # `>=` in the 3-D env
        self.step_count = torch.zeros(n_env, dtype=torch.int64, device=self.device)
        self._seed = 0
        self._n_autoreset = 0

    def _draws(self, env_ids, initial):
        # reset(seed): env i == a reference env reset with seed + global index; autoreset: one batched stream
        if initial:
            return np.array([np.random.Generator(np.random.PCG64(np.random.SeedSequence(
                int(self._seed + self.env_offset + i)))).uniform(-1.0, 1.0) for i in env_ids])
        self._n_autoreset += 1
        ss = np.random.SeedSequence([int(self._seed), int(self.env_offset), int(self._n_autoreset)])
        return np.random.Generator(np.random.PCG64(ss)).uniform(-1.0, 1.0, len(env_ids))

    def reset(self, seed: int = 0):
        torch = self.torch
        self._seed = seed
        self._n_autoreset = 0
        init = torch.as_tensor(pendulum3d_init_params(self._draws(range(self.n_env), True)), device=self.device)
        self.handle.reset(init.contiguous())
        self.step_count.zero_()
        self.handle.observe(None, self.obs)
        return self.obs.clone(), {}

    def step(self, action):
        torch = self.torch
        action = action.to(device=self.device, dtype=torch.float32).reshape(self.n_env, 2).contiguous()
        self.handle.step(action, self.step_skip, self.obs, self.reward, self.terminated)
        self.step_count += 1
        truncated = self.step_count >= self._first_truncated
        terminated = self.terminated.bool()
        obs, reward = self.obs.clone(), self.reward.clone()
        info = {"time": torch.as_tensor(self._time_table, device=self.device)[
            self.step_count.clamp(max=len(self._time_table) - 1)], "tilt": self.handle.aux_tensor()[:, 6].clone()}
        done = terminated | truncated
        if self.autoreset and bool(done.any()):
            idx = torch.nonzero(done).flatten()
            ids = idx.cpu().numpy()
            info["final_obs"], info["reset_idx"] = obs[idx].clone(), idx
            init = torch.as_tensor(pendulum3d_init_params(self._draws(ids, False)), device=self.device)
            self.handle.reset(init.contiguous(), idx.to(torch.int32).contiguous())
            self.step_count[idx] = 0
            fresh = torch.empty_like(self.obs)
            self.handle.observe(None, fresh)
            obs[idx] = fresh[idx]
        return obs, reward, terminated, truncated, info

    def fields(self):
        return self.handle.fields()

    def close(self):
        self.handle.close()
