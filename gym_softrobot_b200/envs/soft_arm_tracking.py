"""SoftArmTracking-v0 on the B200 kernel.

Host-side mirror of `/root/reference/gym_softrobot/envs/soft_arm/soft_arm_tracking.py`
(`SoftArmTrackingEnv`, lines 101-487): a clamped arm (n=40, L=1000 mm, `OneEndFixedBC`,
`AnalyticalLinearDamper`) bends under two `MuscleTorquesWithVaryingBetaSplines` forcings (normal and
binormal direction, 4 control values each, `utils/custom_elastica/muscle_torque/
muscle_torques_with_bspline.py`) to bring its tip to a target that is either fixed (game_mode 1) or
moves along a seeded trajectory (game_mode 2, lines 44-98).  One env-step is 50 PositionVerlet substeps
(line 218) = one `sr_step` launch; the spline re-fit at the current element lengths happens inside the
kernel.  The target `Sphere` carries no load and is overwritten every substep (lines 223-224), so only
its value at the step boundary is observable: it lives on the host side as a table.
"""
from typing import Optional

import numpy as np

from .. import _native as nat
from .fork import ForkableVectorEnv
from ..compat import Box, Env
from .soft_pendulum import _advance_time

_N_ELEM, _DT, _L, _R, _E = 40, 2.0e-4, 1000.0, 50.0, 2e6
_N_CTRL = 4
_UPDATE = int(np.rint(0.01 / _DT))          # substeps per env-step
_FINAL_TIME = 5.0


def target_trajectory(final_time, sim_dt, v_scale, rng):
    """Moving target of game_mode 2 (`generate_trajectory`, soft_arm_tracking.py:44-98): per axis a product
    of three sines with seeded frequencies; same draw order and floating-point expression order."""
    end_time = final_time * 1.1
    numpoints = np.rint(1 / sim_dt * end_time).astype(int)
    t = end_time * np.arange(numpoints, dtype=np.float64) / (numpoints - 1)
    t += rng.random() * 3600
    out = np.zeros((numpoints, 3))
    for axis, amp in enumerate((0.8, 0.4, 0.8)):
        f1, f2, f3 = (rng.uniform(2, 5) * 0.025 * v_scale for _ in range(3))
        sign = rng.integers(0, 2) * 2 - 1
        out[:, axis] = (sign * amp * np.sin(2 * np.pi * f1 * t) * np.sin(2 * np.pi * f2 * t)
                        * np.sin(2 * np.pi * f3 * t) * 1000)
        if axis == 1:
            out[:, 1] += 0.4
    return out


def substeps_per_step(time_step):
    """Substeps per env-step: the reference's 0.01 s of simulated time per env-step (50 at its 2e-4 s step)."""
    return int(np.rint(0.01 / time_step))


def truncation_steps(update, time_step, final_time=_FINAL_TIME):
    """Env-steps after which an episode is truncated: the first k with `tick * sim_dt >= final_time`, tick = k * update
    substeps as an integer and the product in float64, as the reference evaluates it (soft_arm_tracking.py:254)."""
    k = max(1, int(final_time / (update * time_step)) - 1)
    while k > 1 and (k - 1) * update * time_step >= final_time:
        k -= 1
    while not (k * update * time_step >= final_time):
        k += 1
    return k


def spline_scale(n_elems):
    """Spline torque magnitude per element: the reference's 10 R E at its 40 elements, times 40 / n_elems, so that the
    torque summed over the arm does not grow with refinement (exactly the reference's value at n_elems = 40)."""
    return 10 * _R * _E * (_N_ELEM / n_elems)


def _make_handle(n_env, device, dtype=nat.DTYPE_F64, n_elems=_N_ELEM, time_step=_DT):
    return nat.Handle(
        model=nat.MODEL_ROD, n_env=n_env, n_elem=n_elems, dt=time_step, base_length=_L, base_radius=_R,
        density=1000 * 1e-6, youngs_modulus=_E, damping_constant=_E * 1e-7 * 1, bc_kind=nat.BC_ONE_END_FIXED,
        damping_before_constraints=True,          # dampen() is called before constrain() (lines 300-309)
        device=device, dtype=dtype,
        spline=dict(directions=(0, 1), n_ctrl=_N_CTRL, scale=spline_scale(n_elems), max_rate=float("inf")))


class SoftArmTrackingVectorEnv(ForkableVectorEnv):
    """N independent SoftArmTracking-v0 envs (torch CUDA I/O, float64), one physics launch per env-step.

    `n_elems` (3-4095; 1024 and more step on thread-block clusters) and `time_step` refine the arm.  An env-step stays
    0.01 s of simulated time, rint(0.01 / time_step) substeps, and truncation follows `tick * sim_dt >= 5`.  The spline
    torque is applied per element, so a finer arm would feel a larger total torque: the magnitude is scaled by
    40 / n_elems (spline_scale), 1.0 at the reference's 40 elements.  With the reference's unscaled magnitude a
    2048-element arm diverges within its first env-step at 5e-6 s and at 2.5e-6 s; scaled, it tracks a 1024-element arm
    at 1e-5 s to 0.02 mm at the tip after three env-steps of random targets (longer horizons not checked).  A finer arm
    needs a smaller step: 5e-6 s at 2048 elements."""

    PER_ENV = ("tick", "_targets")   # per-env host state (copy_envs)

    def __init__(self, n_env, game_mode: int = 1, device: int = 0, autoreset: bool = True, n_elems: int = _N_ELEM,
                 time_step: float = _DT):
        import torch
        self.torch = torch
        self.n_env, self.mode = n_env, game_mode
        self.n_elems, self.time_step = n_elems, time_step
        self.update = substeps_per_step(time_step)
        self.device = torch.device(f"cuda:{device}")
        self.autoreset = autoreset
        self.single_action_space = Box(-1.0, 1.0, shape=(2 * _N_CTRL,), dtype=np.float64)
        self.single_observation_space = Box(-np.inf, np.inf, shape=(_N_CTRL * 2 + 6,), dtype=np.float64)
        self.handle = _make_handle(n_env, device, n_elems=n_elems, time_step=time_step)
        self._scratch = (torch.empty((n_env, 6), dtype=torch.float32, device=self.device),
                         torch.empty(n_env, dtype=torch.float64, device=self.device),
                         torch.empty(n_env, dtype=torch.uint8, device=self.device))
        self._init = np.zeros((1, 9)); self._init[0, 4] = 1.0; self._init[0, 8] = 1.0   # direction +y, normal +z
        # tick -> truncated: `self.tick * self.sim_dt >= 5` evaluated in float64 as the reference does
        self.n_updates = truncation_steps(self.update, time_step)
        self._targets = torch.zeros((n_env, self.n_updates + 1, 3), dtype=torch.float64, device=self.device)
        self.tick = torch.zeros(n_env, dtype=torch.int64, device=self.device)      # in env-steps
        self._seq = None

    # -- helpers -----------------------------------------------------------------------------
    def _target_now(self):
        idx = self.tick.clamp(max=self.n_updates)
        return self._targets[self.torch.arange(self.n_env, device=self.device), idx]

    def _state(self):
        # get_state (lines 159-209): 4 segment means of kappa[0] and kappa[1], tip position, target
        torch = self.torch
        f = self.handle.fields()
        kap = f["kappa"]                                     # stale, as in the reference (SURVEY A.6)
        seg = int((self.n_elems - 1) / _N_CTRL)
        parts = []
        for c in (0, 1):
            m = [kap[:, c, seg * i:seg * (i + 1)].mean(dim=1) for i in range(_N_CTRL - 1)]
            m.append(kap[:, c, seg * (_N_CTRL - 1):].mean(dim=1))
            parts.append(torch.stack(m, dim=1) * _L / (2 * np.pi))
        tip = f["position_collection"][:, :, -1] / _L
        return torch.cat([parts[0], parts[1], tip, self._target_now() / 1000], dim=1)

    def _new_targets(self, idx, seed):
        torch = self.torch
        if self.mode == 1:
            self._targets[idx] = torch.tensor([500.0, 500.0, 500.0], dtype=torch.float64, device=self.device)
            return
        if self._seq is None or seed is not None:
            self._seq = np.random.SeedSequence(seed)
        rows = []
        for _ in range(len(idx)):                            # one independent stream per episode
            rng = np.random.Generator(np.random.PCG64(self._seq.spawn(1)[0]))
            w = target_trajectory(_FINAL_TIME, self.time_step, 0.1, rng)
            rows.append(w[::self.update][:self.n_updates + 1])
        self._targets[idx] = torch.as_tensor(np.stack(rows), device=self.device)

    def _reset_envs(self, idx=None, seed=None, new_targets=True):
        torch = self.torch
        n = self.n_env if idx is None else int(idx.numel())
        init = torch.as_tensor(np.repeat(self._init, n, axis=0), device=self.device).contiguous()
        self.handle.reset(init, None if idx is None else idx.to(torch.int32).contiguous())
        all_idx = torch.arange(self.n_env, device=self.device) if idx is None else idx
        if new_targets:     # (the single-env facade supplies the trajectory from its own generator)
            self._new_targets(all_idx, seed)
        self.tick[all_idx] = 0

    # -- API ---------------------------------------------------------------------------------
    def reset(self, seed: Optional[int] = None):
        self._reset_envs(None, seed)
        return self._state(), {}

    def step(self, action):
        torch = self.torch
        action = action.to(device=self.device, dtype=torch.float64).reshape(self.n_env, 2 * _N_CTRL)
        pts, _ = self.handle.spline_tensors()
        pts[:, 0, :_N_CTRL] = action[:, :_N_CTRL]           # spline_points_func_array_normal_dir[:] = ...
        pts[:, 1, :_N_CTRL] = action[:, _N_CTRL:]
        obs6, rew, term = self._scratch
        self.handle.step(None, self.update, obs6, rew, term)
        self.tick += 1
        tip = self.handle.fields()["position_collection"][:, :, -1]
        tip_to_target = (self._target_now() - tip) / 1000
        reward = -tip_to_target.norm(dim=1).square()
        state = self._state()
        invalid = torch.isnan(state).any(dim=1)
        reward = torch.where(invalid, torch.full_like(reward, -100.0), reward)
        state = torch.nan_to_num(state)
        terminated = invalid
        truncated = self.tick >= self.n_updates
        info = {}
        done = terminated | truncated
        if self.autoreset and bool(done.any()):
            idx = torch.nonzero(done).flatten()
            info["final_obs"], info["reset_idx"] = state[idx].clone(), idx
            self._reset_envs(idx)
            state[idx] = self._state()[idx]
        return state, reward, terminated, truncated, info

    def fields(self):
        return self.handle.fields()

    def close(self):
        self.handle.close()


class SoftArmTrackingEnv(Env):
    """Drop-in for the reference `SoftArmTrackingEnv` (same kwargs, lines 104-157): a batch of one."""

    metadata = {"render_modes": ["rgb_array", "human"], "render_fps": 30}

    def __init__(self, game_mode: int = 1, render_mode: Optional[str] = None, device: int = 0):
        super().__init__()
        if render_mode not in {None, *self.metadata["render_modes"]}:
            raise ValueError(f"Unsupported render mode: {render_mode}")
        self.render_mode = render_mode
        self.mode = game_mode
        self._vec = SoftArmTrackingVectorEnv(1, game_mode, device, autoreset=False)
        self.action_space = self._vec.single_action_space
        self.observation_space = self._vec.single_observation_space
        self.n_elem, self.sim_dt, self.num_steps_per_update = _N_ELEM, _DT, _UPDATE
        self.time_tracker = np.float64(0.0)
        self.tick = 0

    def reset(self, *, seed: Optional[int] = None, options: Optional[dict] = None):
        super().reset(seed=seed)
        # the trajectory draws come from the env's own generator, right after reset(seed) (line 412-418)
        if self.mode == 2:
            v = self._vec
            v._reset_envs(None, None, new_targets=False)
            w = target_trajectory(_FINAL_TIME, _DT, 0.1, self.np_random)
            v._targets[0] = v.torch.as_tensor(w[::_UPDATE][:v.n_updates + 1], device=v.device)
            obs = v._state()
        else:
            obs, _ = self._vec.reset()
        self.time_tracker = np.float64(0.0)
        self.tick = 0
        self._target = self._vec._targets[0, 0].cpu().numpy()
        return obs[0].cpu().numpy(), {}

    def step(self, action):
        import torch
        a = torch.as_tensor(np.asarray(action, dtype=np.float64).reshape(1, -1), device=self._vec.device)
        obs, reward, term, trunc, _ = self._vec.step(a)
        self.time_tracker = _advance_time(self.time_tracker, _DT, _UPDATE)
        self.tick += _UPDATE
        if bool(term[0]):
            print("Episode blew up. Maybe try a smaller dt?")
        if bool(trunc[0]):
            print("Episode has reached max time")
        self._target = self._vec._target_now()[0].cpu().numpy()
        r = reward[0].item()
        return (obs[0].cpu().numpy(), -100 if bool(term[0]) else r, bool(term[0]), bool(trunc[0]),
                {"ctime": self.time_tracker})

    def rod_state(self):
        return {k: v[0].cpu().numpy() for k, v in self._vec.fields().items()}

    def render(self):
        return None

    def close(self):
        self._vec.close()
