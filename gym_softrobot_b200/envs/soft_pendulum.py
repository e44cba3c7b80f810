"""SoftPendulum-v0 on the B200 kernel.

Host-side mirror of `/root/reference/gym_softrobot/envs/soft_pendulum/soft_pendulum.py`
(`SoftPendulumEnv`, lines 45-251) and `.../soft_pendulum/build.py:29-115`
(`build_soft_pendulum`): same constructor kwargs, spaces, seeding, reward,
termination and `info`.  The substep loop (`soft_pendulum.py:183-184`) is one
`sr_step` launch of the fused kernel; there is no CPU fallback.

Two façades over the same C-ABI handle:
  * `SoftPendulumEnv`        single env, Gymnasium API, host (NumPy) I/O  — drop-in
  * `SoftPendulumVectorEnv`  N envs, torch CUDA tensors in / out, same-step autoreset
"""
from typing import Optional

import numpy as np

from .. import _native as nat
from .fork import ForkableVectorEnv
from ..compat import Box, Env

# defaults of the reference build function (soft_pendulum/build.py:19-26)
_PENDULUM_PROPERTIES = {"youngs_modulus": 1e6, "density": 1000.0}
_DEFAULT_SCALE_LENGTH = {"base_length": 1.0, "base_radius": 0.05}
_GRAVITY = (0.0, -9.80665, 0.0)   # build.py:88-91
_DAMPING_CONSTANT = 2e-3          # build.py:108-113


def pendulum_init_params(u01):
    """start / direction / normal rows for `sr_reset`, from the uniform draw(s) `u01`.

    Exactly the host arithmetic of build.py:46-51 (NumPy float64), so the initial
    directors are bit-identical to the reference's.
    """
    u01 = np.atleast_1d(np.asarray(u01, dtype=np.float64))
    theta = np.deg2rad(90 + (u01 - 0.5) * 10)
    init = np.zeros((u01.shape[0], 9))
    init[:, 3] = 1.0 * np.cos(theta)
    init[:, 4] = 1.0 * np.sin(theta)
    init[:, 6] = 1.0 * np.sin(theta)
    init[:, 7] = -1.0 * np.cos(theta)
    return init


def _make_handle(n_env, n_elems, time_step, device, math, dtype=nat.DTYPE_F64):
    return nat.Handle(
        model=nat.MODEL_SOFT_PENDULUM, n_env=n_env, n_elem=n_elems, dt=time_step,
        gravity=_GRAVITY, damping_constant=_DAMPING_CONSTANT, bc_kind=nat.BC_PENDULUM_SLIDER,
        point_force_on_base=True, damping_before_constraints=False, device=device, math=math, dtype=dtype,
        **_DEFAULT_SCALE_LENGTH, **_PENDULUM_PROPERTIES,
    )


def _advance_time(t, time_step, n_substeps):
    """PositionVerlet adds dt/2 twice per substep to a float64 (SURVEY B-5); `n*dt` would differ."""
    half = 0.5 * time_step
    for _ in range(n_substeps):
        t = t + half
        t = t + half
    return t


class SoftPendulumEnv(Env):
    """Drop-in for the reference `SoftPendulumEnv` (same kwargs; soft_pendulum.py:59-67)."""

    metadata = {"render_modes": ["rgb_array"], "render_fps": 25}

    def __init__(self, final_time=5.0, time_step=1.0e-4, recording_fps=25, n_elems=50,
                 config_generate_video=False, render_mode: Optional[str] = None, device: int = 0,
                 math: int = nat.MATH_FAST):
        super().__init__()
        if render_mode not in {None, *self.metadata["render_modes"]}:
            raise ValueError(f"Unsupported render mode: {render_mode}")
        self.render_mode = render_mode
        self.final_time = final_time
        self.time_step = time_step
        self.total_steps = int(self.final_time / self.time_step)
        self.recording_fps = recording_fps
        self.step_skip = int(1.0 / (recording_fps * time_step))
        self.n_elems = n_elems
        self.n_seg = n_elems - 1
        self.n_action = 1
        self.action_space = Box(np.ones(1) * (-22), np.ones(1) * 22, shape=(1,), dtype=np.float32)
        self.observation_space = Box(-np.inf, np.inf, shape=(4,), dtype=np.float32)
        self.reward_range = 100.0
        self._prev_action = np.zeros(1, dtype=np.float32)
        self.config_generate_video = config_generate_video
        self._device, self._math = device, math
        self._handle = None
        self.time = np.float64(0.0)
        self.counter = 0

    # ------------------------------------------------------------------ API
    def reset(self, *, seed: Optional[int] = None, options: Optional[dict] = None):
        super().reset(seed=seed)
        if self._handle is None:
            self._handle = _make_handle(1, self.n_elems, self.time_step, self._device, self._math)
        # build.py:47-49 draws one uniform from the env generator
        init = pendulum_init_params(self.np_random.random())
        self._handle.reset_host(init)
        # NB the reference does not clear `_prev_action` in reset (soft_pendulum.py:108-147); neither do we
        self.time = np.float64(0.0)
        self.counter = 0
        return self.get_state(), {}

    def get_state(self):
        import torch
        dev = f"cuda:{self._device}"
        obs = torch.empty((1, 4), dtype=torch.float32, device=dev)
        pa = torch.as_tensor(self._prev_action, device=dev).reshape(1, 1).contiguous()
        self._handle.observe(pa, obs)
        return obs.cpu().numpy()[0]

    def step(self, action):
        a = np.asarray(action, dtype=np.float32).reshape(1)
        self._prev_action[:] = a
        obs, reward, terminated = self._handle.step_host(a.reshape(1, 1), self.step_skip)
        self.time = _advance_time(self.time, self.time_step, self.step_skip)
        term = bool(terminated[0])
        if term:
            print(f" Nan detected in, exiting simulation now. {self.time=}")
        timelimit = bool(self.time > self.final_time)
        info = {"time": self.time, "TimeLimit.truncated": timelimit}
        self.counter += 1
        return obs[0].copy(), np.float64(reward[0]), term, timelimit, info

    # reference-named rod views (position_collection, tangents, ...), NumPy copies
    def rod_state(self):
        return {k: v[0].cpu().numpy() for k, v in self._handle.fields().items()}

    def render(self):
        return None  # rendering is out of scope (SURVEY §2 row 15)

    def close(self):
        if self._handle is not None:
            self._handle.close()
            self._handle = None


class SoftPendulumVectorEnv(ForkableVectorEnv):
    """N independent SoftPendulum-v0 envs stepped by one kernel launch per env-step.

    Observations / rewards / flags are torch tensors on the GPU; actions are a
    float32 CUDA tensor [n_env, 1].  Env i is seeded like a reference env reset with
    `seed + i` (`PCG64(SeedSequence(seed + i))`, build.py:47-49).  Envs that finish
    are reset inside the same `step` call (final observation returned in
    `info["final_obs"]`).
    """

    PER_ENV = ("step_count", "prev_action")   # per-env host state (copy_envs)

    def __init__(self, n_env, final_time=5.0, time_step=1.0e-4, recording_fps=25, n_elems=50,
                 device: int = 0, math: int = nat.MATH_FAST, autoreset: bool = True,
                 env_offset: int = 0, dtype: str = "float64"):
        import torch
        self.torch = torch
        self.n_env, self.n_elems = n_env, n_elems
        self.final_time, self.time_step = final_time, time_step
        self.step_skip = int(1.0 / (recording_fps * time_step))
        self.device = torch.device(f"cuda:{device}")
        self.env_offset = env_offset  # global index of env 0 (multi-GPU sharding)
        self.autoreset = autoreset
        self.single_action_space = Box(np.ones(1) * (-22), np.ones(1) * 22, shape=(1,), dtype=np.float32)
        self.single_observation_space = Box(-np.inf, np.inf, shape=(4,), dtype=np.float32)
        # FP64 matches PyElastica (1e-9); "float32" is the optional fast mode (state to ~1e-4)
        self.handle = _make_handle(n_env, n_elems, time_step, device, math,
                                   nat.DTYPE_F32 if dtype == "float32" else nat.DTYPE_F64)
        self.obs = torch.empty((n_env, 4), dtype=torch.float32, device=self.device)
        self.reward = torch.empty(n_env, dtype=torch.float64, device=self.device)
        self.terminated = torch.empty(n_env, dtype=torch.uint8, device=self.device)
        # time after j env-steps, accumulated exactly like the reference
        n_max = int(final_time / (self.step_skip * time_step)) + 8
        table, t = [np.float64(0.0)], np.float64(0.0)
        for _ in range(n_max):
            t = _advance_time(t, time_step, self.step_skip)
            table.append(t)
        self._time_table = np.array(table)
        self._first_truncated = int(np.argmax(self._time_table > final_time))
        self.step_count = torch.zeros(n_env, dtype=torch.int64, device=self.device)
        # like the reference env (soft_pendulum.py:97,108-147,165) the previous action is set at construction and by
        # step() only: the observation right after a reset still carries the last action of the episode before
        self.prev_action = torch.zeros((n_env, 1), dtype=torch.float32, device=self.device)
        self._seed = 0
        self._n_autoreset = 0

    def _draws(self, env_ids, initial):
        """Uniform draws behind the initial angle (build.py:47-49).  At reset(seed) env i draws from
        PCG64(SeedSequence(seed + global_index)) — exactly a reference env reset with that seed; re-draws
        at autoreset come from one batched stream keyed by (seed, shard offset, reset counter)."""
        if initial:
            return np.array([np.random.Generator(np.random.PCG64(np.random.SeedSequence(
                int(self._seed + self.env_offset + i)))).random() for i in env_ids])
        self._n_autoreset += 1
        ss = np.random.SeedSequence([int(self._seed), int(self.env_offset), int(self._n_autoreset)])
        return np.random.Generator(np.random.PCG64(ss)).random(len(env_ids))

    def reset(self, seed: int = 0):
        torch = self.torch
        self._seed = seed
        self._n_autoreset = 0
        init = torch.as_tensor(pendulum_init_params(self._draws(range(self.n_env), True)), device=self.device)
        self.handle.reset(init.contiguous())
        self.step_count.zero_()
        self.handle.observe(self.prev_action, self.obs)
        return self.obs.clone(), {}

    def step(self, action):
        torch = self.torch
        action = action.to(device=self.device, dtype=torch.float32).reshape(self.n_env, 1).contiguous()
        self.handle.step(action, self.step_skip, self.obs, self.reward, self.terminated)
        self.prev_action = action
        self.step_count += 1
        truncated = self.step_count >= self._first_truncated
        terminated = self.terminated.bool()
        obs, reward = self.obs.clone(), self.reward.clone()
        info = {"time": torch.as_tensor(self._time_table, device=self.device)[
            self.step_count.clamp(max=len(self._time_table) - 1)]}
        done = terminated | truncated
        if self.autoreset and bool(done.any()):
            idx = torch.nonzero(done).flatten()
            ids = idx.cpu().numpy()
            info["final_obs"] = obs[idx].clone()
            info["reset_idx"] = idx
            init = torch.as_tensor(pendulum_init_params(self._draws(ids, False)), device=self.device)
            self.handle.reset(init.contiguous(), idx.to(torch.int32).contiguous())
            self.step_count[idx] = 0
            fresh = torch.empty_like(self.obs)
            self.handle.observe(self.prev_action, fresh)
            obs[idx] = fresh[idx]
        return obs, reward, terminated, truncated, info

    def fields(self):
        return self.handle.fields()

    def close(self):
        self.handle.close()
