"""ContinuumSnake-v0 on the B200 kernel.

Host-side mirror of `/root/reference/gym_softrobot/envs/snake/continuum_snake.py` (`ContinuumSnakeEnv`,
lines 134-379): one free rod (n=50, L=0.35 m) on a plane with anisotropic kinetic friction, gravity,
`AnalyticalLinearDamper(1e-4)`, driven by PyElastica's travelling-wave `MuscleTorques` whose B-spline
amplitude beta(s) and wave number are rebuilt from the 7-dim action (lines 186-198).  One env-step is
25 000 PositionVerlet substeps of 8e-6 s (lines 283-291); the reward is the period-averaged forward
velocity computed from callback samples taken every 2083 substeps (lines 40-101, 115-131, 352-356).

The substeps run inside `sr_step`; launches are cut at the callback substeps so the samples are read
from the state views exactly where the reference's callback fires.
"""
from typing import Optional

import numpy as np

from .. import _native as nat
from .fork import ForkableVectorEnv
from ..compat import Box, Env

_L0 = 0.35
_G = -9.80665


def snake_contact_params(period=2.0, before_forcing=False):
    """Plane + friction of `_build` (continuum_snake.py:339-357): kinetic friction only, k=1, nu=1e-6."""
    froude = 0.1
    mu = _L0 / (period * period * np.abs(_G) * froude)
    return dict(plane_origin=[0.0, -_L0 * 0.011, 0.0], plane_normal=[0.0, 1.0, 0.0], k=1.0, nu=1e-6,
                slip_velocity_tol=1e-8, static_mu=np.zeros(3), kinetic_mu=np.array([mu, 1.5 * mu, 2.0 * mu]),
                before_forcing=before_forcing)


def beta_spline_matrix(n_coeff, n_elem):
    """`_bspline(b)(s)` of PyElastica (clamped cubic B-spline through `n_coeff` control values, zero
    end coefficients) evaluated at s_k = cumsum(rest_lengths)_k / L is linear in b: [n_elem, n_coeff]."""
    from scipy.interpolate import BSpline
    pts = np.linspace(0.0, 1.0, n_coeff)
    knots = np.hstack((np.zeros(3), pts, np.ones(3)))
    s = np.cumsum(np.full(n_elem, _L0 / n_elem))
    s /= s[-1]
    cols = []
    for k in range(n_coeff):
        c = np.zeros(n_coeff + 2); c[k + 1] = 1.0
        cols.append(BSpline(knots, c, 3, extrapolate=False)(s))
    return np.stack(cols, axis=1)


def projected_forward_velocity(times, com, vel, period):
    """`compute_projected_velocity` (continuum_snake.py:40-101), batched over envs: `times` [S] (host),
    `com` / `vel` [n_env, S, 3] torch tensors of the callback samples; returns the period-averaged
    forward velocity [n_env] (0 until three periods have been sampled)."""
    import torch
    zero = torch.zeros(com.shape[0], dtype=com.dtype, device=com.device)
    tpp = np.asarray(times) / period
    if len(tpp) < 2:
        return zero
    P = int(1.0 / (tpp[-1] - tpp[-2]))          # samples per period
    n_period = int(tpp[-1])
    if n_period - 2 <= 0:
        return zero
    shifts = [(com[:, (i + 1) * P:(i + 2) * P] - com[:, i * P:(i + 1) * P]).mean(dim=1)
              for i in range(1, n_period - 1)]
    direction = torch.stack(shifts, dim=1).mean(dim=1)
    direction = direction / direction.norm(dim=1, keepdim=True)
    mag = (vel * direction[:, None, :]).sum(dim=2)                    # [n_env, S]
    along = mag[:, :, None] * direction[:, None, :]
    return along[:, 2 * P:].mean(dim=1)[:, 2]


class ContinuumSnakeVectorEnv(ForkableVectorEnv):
    """N independent ContinuumSnake-v0 envs (torch CUDA I/O); they advance in lockstep (the reference
    env never terminates early, so every env truncates at the same step)."""

    PER_ENV = ("_com", "_vel")   # per-env host state (copy_envs)

    period = 2.0
    time_step = 8e-6
    n_elems = 50

    def __init__(self, n_env, device: int = 0, autoreset: bool = True, dtype=nat.DTYPE_F64):
        import torch
        self.torch = torch
        self.n_env = n_env
        self.device = torch.device(f"cuda:{device}")
        self.autoreset = autoreset
        self.final_time = (11.0 + 0.01) * self.period
        self.step_skip = int(1.0 / (5 * self.time_step))                 # rendering_fps = 5
        self.callback_step_skip = int(1.0 / (60 * self.time_step))
        lo, hi = -np.ones(7) * 1e-2, np.ones(7) * 1e-2
        lo[-1], hi[-1] = 0.5, 3.0
        self.single_action_space = Box(lo, hi, dtype=np.float32)
        n = self.n_elems
        self.single_observation_space = Box(-np.inf, np.inf, shape=((n + 1) * 3 * 2 + n * 9,), dtype=np.float32)
        E = 1e6
        self.handle = nat.Handle(
            model=nat.MODEL_ROD, n_env=n_env, n_elem=n, dt=self.time_step, base_length=_L0,
            base_radius=_L0 * 0.011, density=1000.0, youngs_modulus=E, shear_modulus=E / (0.5 + 1.0),
            gravity=(0.0, _G, 0.0), damping_constant=1e-4, bc_kind=nat.BC_FREE, device=device, dtype=dtype,
            contact=snake_contact_params(self.period),
            muscle=dict(period=self.period, ramp_up_time=self.period, phase_shift=0.0, direction=(0.0, 1.0, 0.0)))
        self._W = torch.as_tensor(beta_spline_matrix(6, n), device=self.device)      # [50, 6] f64
        m = np.full(n + 1, 1.0); m[0] = m[-1] = 0.5
        self._mass_w = torch.as_tensor(m / m.sum(), device=self.device)
        self._scratch = (torch.empty((n_env, 6), dtype=torch.float32, device=self.device),
                         torch.empty(n_env, dtype=torch.float64, device=self.device),
                         torch.empty(n_env, dtype=torch.uint8, device=self.device))
        self._init = np.zeros((1, 9)); self._init[0, 5] = 1.0; self._init[0, 7] = 1.0   # direction +z, normal +y
        n_samples = int(self.final_time / self.time_step) // self.callback_step_skip + 16
        self._com = torch.zeros((n_env, n_samples, 3), dtype=torch.float64, device=self.device)
        self._vel = torch.zeros_like(self._com)
        self._times = []
        self._substeps = 0
        self._clock = np.float64(0.0)

    # -- helpers -----------------------------------------------------------------------------
    def _sample(self):
        # ContinuumSnakeCallBack.make_callback (continuum_snake.py:115-131)
        f = self.handle.fields()
        k = len(self._times)
        if k >= self._com.shape[1]:      # stepping past the time limit without a reset (the reference keeps going too)
            grow = self.torch.zeros_like(self._com)
            self._com, self._vel = self.torch.cat([self._com, grow], dim=1), self.torch.cat([self._vel, grow], dim=1)
        self._com[:, k] = (f["position_collection"] * self._mass_w).sum(dim=2)
        self._vel[:, k] = (f["velocity_collection"] * self._mass_w).sum(dim=2)
        self._times.append(float(self._clock))      # host mirror of the in-kernel clock: no device read-back per sample

    def _advance_clock(self, n_substeps):
        # the kernel (and PositionVerlet) advance time by dt/2 twice per substep; cumsum adds left to right, so this
        # is that very sequence of float64 additions
        self._clock = np.cumsum(np.concatenate([[self._clock], np.full(2 * n_substeps, 0.5 * self.time_step)]))[-1]

    def _obs(self):
        f = self.handle.fields()
        n = self.n_env
        return self.torch.cat([f["position_collection"].reshape(n, -1), f["velocity_collection"].reshape(n, -1),
                               f["director_collection"].reshape(n, -1)], dim=1).float()

    def _check_copy_source(self, src):
        # the envs of a batch share one host clock and sample history: envs of another batch continue here only
        # from the same instant
        if src is not self and (src._clock != self._clock or src._substeps != self._substeps or src._times != self._times):
            raise ValueError("copy_envs: a ContinuumSnake env continues only in a vector env at the same clock "
                             f"(src at t = {float(src._clock)}, {src._substeps} substeps; here t = {float(self._clock)}, "
                             f"{self._substeps} substeps)")

    def _projected_velocity(self):
        S = len(self._times)
        return projected_forward_velocity(np.array(self._times), self._com[:, :S], self._vel[:, :S], self.period)

    # -- API ---------------------------------------------------------------------------------
    def reset(self, seed: int = 0):
        torch = self.torch
        init = torch.as_tensor(np.repeat(self._init, self.n_env, axis=0), device=self.device).contiguous()
        self.handle.reset(init, None)
        mu = self.handle.muscle_tensor()
        mu.zero_()
        mu[:, 1] = float(np.float32(2.0 * np.pi) / np.float32(1.0))       # _build: b_coeff = 0, wave_length = 1
        self._times, self._substeps, self._clock = [], 0, np.float64(0.0)
        self._sample()                                                     # the callback's finalize-time sample
        return self._obs(), {}

    def step(self, action):
        torch = self.torch
        action = action.to(device=self.device, dtype=torch.float32).reshape(self.n_env, 7)
        # set_action (continuum_snake.py:186-198): beta spline through the six coefficients, float32 wave number
        mu = self.handle.muscle_tensor()
        b = action[:, :6].double()
        beta = b[:, 0:1] * self._W[:, 0]
        for k in range(1, 6):
            beta = beta + b[:, k:k + 1] * self._W[:, k]
        mu[:, 2:] = beta
        mu[:, 1] = (torch.tensor(2.0 * np.pi, dtype=torch.float32, device=self.device) / action[:, 6]).double()
        obs6, rew, term = self._scratch
        left = self.step_skip
        while left > 0:
            k = min(left, self.callback_step_skip - self._substeps % self.callback_step_skip)
            self.handle.step(None, k, obs6, rew, term)
            self._advance_clock(k)
            self._substeps += k
            left -= k
            if self._substeps % self.callback_step_skip == 0:
                self._sample()
        reward = self._projected_velocity()
        time = mu[:, 0].clone()
        truncated = time >= self.final_time
        terminated = torch.zeros(self.n_env, dtype=torch.bool, device=self.device)
        obs = self._obs()
        info = {"time": time}
        if self.autoreset and bool(truncated.any()):
            info["final_obs"] = obs.clone()
            obs, _ = self.reset()
        return obs, reward, terminated, truncated, info

    def fields(self):
        return self.handle.fields()

    def close(self):
        self.handle.close()


class ContinuumSnakeEnv(Env):
    """Drop-in for the reference `ContinuumSnakeEnv` (continuum_snake.py:134-219): a batch of one."""

    metadata = {"render_modes": ["rgb_array", "human"], "render_fps": 30}

    def __init__(self, render_mode: Optional[str] = None, device: int = 0):
        super().__init__()
        if render_mode not in {None, *self.metadata["render_modes"]}:
            raise ValueError(f"Unsupported render mode: {render_mode}")
        self.render_mode = render_mode
        self._vec = ContinuumSnakeVectorEnv(1, device, autoreset=False)
        self.action_space = self._vec.single_action_space
        self.observation_space = self._vec.single_observation_space
        self.step_skip, self.period, self.final_time = self._vec.step_skip, self._vec.period, self._vec.final_time
        self.time = np.float64(0.0)

    def reset(self, *, seed: Optional[int] = None, options: Optional[dict] = None):
        super().reset(seed=seed)
        obs, _ = self._vec.reset()
        self.time = np.float64(0.0)
        return obs[0].cpu().numpy(), {}

    def step(self, action):
        import torch
        err_msg = f"{action!r} ({type(action)}) invalid: expected {self.action_space}"
        assert self.action_space.contains(action), err_msg
        a = torch.as_tensor(np.asarray(action, dtype=np.float32).reshape(1, -1), device=self._vec.device)
        obs, reward, term, trunc, info = self._vec.step(a)
        self.time = np.float64(info["time"][0].item())
        return obs[0].cpu().numpy(), reward[0].item(), False, bool(trunc[0]), {}

    def rod_state(self):
        return {k: v[0].cpu().numpy() for k, v in self._vec.fields().items()}

    def render(self):
        return None

    def close(self):
        self._vec.close()
