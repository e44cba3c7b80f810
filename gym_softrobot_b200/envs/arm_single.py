"""OctoArmSingle-v0 on the B200 kernel.

Host-side mirror of `/root/reference/gym_softrobot/envs/octopus/arm_single_env.py` (`ArmSingleEnv`,
lines 41-330) and `build_arm` (`envs/octopus/build.py:220-292`): one free rod (n=50, L=0.35 m) lying on
a frictional plane (`RodPlaneContactWithAnisotropicFriction`), gravity, `AnalyticalLinearDamper(1e-2)`,
actuated through its rest curvature (cubic interpolation of 7 control values, lines 226-235).
The substep loop (lines 247-248) is one `sr_step` launch; observation / reward are small torch
reductions over the SoA state, in the reference's expression order.
"""
from typing import Optional

import numpy as np

from .. import _native as nat
from .fork import ForkableVectorEnv
from ..compat import Box, Env
from .soft_pendulum import _advance_time

_ROD = dict(base_length=0.35, base_radius=0.35 * 0.02, density=1000.0, youngs_modulus=1e6)
_G = -9.81


def arm_contact_params(friction_multiplier=1.0, friction_symmetry=False, before_forcing=False):
    """Plane + friction parameters of build_arm / build_octopus (build.py:173-200, 258-283)."""
    L0, r0 = _ROD["base_length"], _ROD["base_radius"]
    period, froude = 2.0, 0.1
    mu = L0 / (period * period * np.abs(_G) * froude)
    kin = (np.array([mu, mu, mu]) if friction_symmetry else np.array([mu, 1.5 * mu, 2.0 * mu])) * friction_multiplier
    return dict(plane_origin=[0.0, 0.0, -r0], plane_normal=[0.0, 0.0, 1.0], k=1e2, nu=1e1,
                slip_velocity_tol=1e-8, static_mu=2 * kin, kinetic_mu=kin, before_forcing=before_forcing)


def curvature_interp_matrix(n_action, n_seg):
    """`interp1d(linspace(0,1,n_action), a, kind="cubic")(linspace(0,1,n_seg))` is linear in `a`:
    build it once as a [n_seg, n_action] matrix by interpolating identity columns with scipy
    (SURVEY Appendix E) — the per-step scipy call of arm_single_env.py:229-234 becomes one GEMV."""
    from scipy.interpolate import interp1d
    xs, xq = np.linspace(0, 1, n_action), np.linspace(0, 1, n_seg)
    return np.stack([interp1d(xs, np.eye(n_action)[i], kind="cubic", axis=-1)(xq) for i in range(n_action)], axis=1)


def _make_handle(n_env, n_elems, time_step, device, dtype=nat.DTYPE_F64):
    return nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n_elems, dt=time_step, gravity=(0.0, 0.0, _G),
                      damping_constant=1e-2, bc_kind=nat.BC_FREE, damping_before_constraints=False,
                      device=device, dtype=dtype, contact=arm_contact_params(), **_ROD)


class ArmSingleVectorEnv(ForkableVectorEnv):
    """N independent OctoArmSingle-v0 envs (torch CUDA I/O), one physics launch per env-step."""

    PER_ENV = ("step_count", "prev_action", "prev_kappa", "prev_com", "prev_dist")   # per-env host state (copy_envs)

    kappa_range = [-49.33508476187419, 49.33545827754751]
    kappa_rate_range = [-21.063520620377012, 24.664591289161944]

    def __init__(self, n_env, final_time=10.0, time_step=7.0e-5, recording_fps=20, n_elems=50, n_action=7,
                 control_penalty_coeff=0.001, device: int = 0, autoreset: bool = True):
        import torch
        self.torch = torch
        self.n_env, self.n_elems, self.n_seg, self.n_action = n_env, n_elems, n_elems - 1, n_action
        if self.n_seg % 7 != 0:
            raise ValueError("the reference observation reshapes kappa to (7, 7): n_elems - 1 must be 49")
        self.final_time, self.time_step = final_time, time_step
        self.step_skip = int(1.0 / (recording_fps * time_step))
        self.control_penalty_coeff = control_penalty_coeff
        self.device = torch.device(f"cuda:{device}")
        self.autoreset = autoreset
        self.single_action_space = Box(np.ones(n_action) * -22, np.ones(n_action) * 22, shape=(n_action,), dtype=np.float32)
        self.single_observation_space = Box(-np.inf, np.inf, shape=(25,), dtype=np.float32)
        self.handle = _make_handle(n_env, n_elems, time_step, device)
        self._W = torch.as_tensor(curvature_interp_matrix(n_action, self.n_seg), device=self.device)  # [49, 7] f64
        self._scratch = (torch.empty((n_env, 6), dtype=torch.float32, device=self.device),
                         torch.empty(n_env, dtype=torch.float64, device=self.device),
                         torch.empty(n_env, dtype=torch.uint8, device=self.device))
        m = np.full(n_elems + 1, 1.0); m[0] = m[-1] = 0.5   # nodal masses up to a common factor
        self._mass_w = torch.as_tensor(m / m.sum(), device=self.device)
        self._target = torch.tensor([1.0, 0.0], dtype=torch.float64, device=self.device)
        self._init = np.zeros((1, 9)); self._init[0, 3] = 1.0; self._init[0, 8] = 1.0   # dir +x, normal +z
        n_max = int(final_time / (self.step_skip * time_step)) + 8
        table, t = [np.float64(0.0)], np.float64(0.0)
        for _ in range(n_max):
            t = _advance_time(t, time_step, self.step_skip)
            table.append(t)
        self._time_table = np.array(table)
        self._first_truncated = int(np.argmax(self._time_table > final_time))
        self.step_count = torch.zeros(n_env, dtype=torch.int64, device=self.device)
        self.prev_action = torch.zeros((n_env, n_action), dtype=torch.float32, device=self.device)

    # -- helpers -----------------------------------------------------------------------------
    def _com(self):
        # compute_position_center_of_mass()[:2]: sum(m x) / sum(m)
        x = self.handle.fields()["position_collection"]
        return (x[:, :2, :] * self._mass_w).sum(dim=2)

    def _obs(self):
        torch = self.torch
        kappa = self.handle.fields()["kappa"][:, 0, :]                      # rod.kappa[0], stale (A.6)
        rate = kappa - self.prev_kappa
        self.prev_kappa = kappa.clone()
        mk = kappa.reshape(self.n_env, 7, 7).mean(dim=2)
        mr = rate.reshape(self.n_env, 7, 7).mean(dim=2)
        k = (mk - self.kappa_range[0]) / (self.kappa_range[1] - self.kappa_range[0])
        kr = (mr - self.kappa_rate_range[0]) / (self.kappa_rate_range[1] - self.kappa_rate_range[0])
        com = self._com()
        com_rate = com - self.prev_com
        self.prev_com = com.clone()
        tgt = self._target.expand(self.n_env, 2)
        return torch.cat([k, kr, com_rate, self.prev_action.double(), tgt], dim=1).float()

    def _reset_envs(self, idx=None):
        torch = self.torch
        n = self.n_env if idx is None else int(idx.numel())
        init = torch.as_tensor(np.repeat(self._init, n, axis=0), device=self.device).contiguous()
        self.handle.reset(init, None if idx is None else idx.to(torch.int32).contiguous())
        rk = self.handle.rest_kappa_tensor()
        if idx is None:
            rk.zero_()
        else:
            rk[idx] = 0

    def reset(self, seed: int = 0):
        self._reset_envs()
        self.step_count.zero_()
        # (the previous action survives a reset, as in the reference: arm_single_env.py:100,203,227 set it at
        # construction and in step() only)
        self.prev_kappa = self.handle.fields()["kappa"][:, 0, :].clone()
        self.prev_com = self._com().clone()
        obs = self._obs()
        self.prev_dist = (self._com() - self._target).norm(dim=1)
        return obs, {}

    def step(self, action):
        torch = self.torch
        action = action.to(device=self.device, dtype=torch.float32).reshape(self.n_env, self.n_action)
        self.prev_action = action.clone()
        # set_action: rest_kappa[0, :] = cubic interpolation of the 7 control values
        # fixed-order accumulation instead of a GEMM: results must not depend on the batch size
        a64 = action.double()
        kap = a64[:, 0:1] * self._W[:, 0]
        for k in range(1, self.n_action):
            kap = kap + a64[:, k:k + 1] * self._W[:, k]
        self.handle.rest_kappa_tensor()[:, 0, :] = kap
        obs6, rew, term = self._scratch
        self.handle.step(None, self.step_skip, obs6, rew, term)
        self.step_count += 1
        f = self.handle.fields()
        invalid = term.bool() | (f["omega_collection"].reshape(self.n_env, -1).norm(dim=1) > 250)
        control_penalty = self.control_penalty_coeff * action.double().square().mean(dim=1)
        com = self._com()
        dist = (com - self._target).norm(dim=1)
        forward = torch.exp(-dist / 0.35) - 0.096
        goal = (dist < 0.1) & ~invalid
        survive = torch.where(invalid, torch.full_like(dist, -1.0), torch.where(goal, torch.full_like(dist, 5.0), torch.zeros_like(dist)))
        reward = torch.where(invalid, torch.zeros_like(dist), forward) - control_penalty + survive
        self.prev_dist = torch.where(invalid, self.prev_dist, dist)
        terminated = invalid | goal
        truncated = self.step_count >= self._first_truncated
        obs = self._obs()
        info = {"time": torch.as_tensor(self._time_table, device=self.device)[
            self.step_count.clamp(max=len(self._time_table) - 1)]}
        done = terminated | truncated
        if self.autoreset and bool(done.any()):
            idx = torch.nonzero(done).flatten()
            info["final_obs"], info["reset_idx"] = obs[idx].clone(), idx
            self._reset_envs(idx)
            self.step_count[idx] = 0
            self.prev_kappa[idx] = self.handle.fields()["kappa"][idx, 0, :]
            self.prev_com[idx] = self._com()[idx]
            fresh = self._obs()
            obs[idx] = fresh[idx]
            self.prev_dist[idx] = (self._com()[idx] - self._target).norm(dim=1)
        return obs, reward, terminated, truncated, info

    def fields(self):
        return self.handle.fields()

    def close(self):
        self.handle.close()


class ArmSingleEnv(Env):
    """Drop-in for the reference `ArmSingleEnv` (same kwargs; arm_single_env.py:55-66): a batch of one."""

    metadata = {"render_modes": ["rgb_array", "human"], "render_fps": 20}

    def __init__(self, final_time=10.0, time_step=7.0e-5, recording_fps=20, n_elems=50, n_action=7,
                 control_penalty_coeff=0.001, config_generate_video=False, policy_mode="centralized",
                 render_mode: Optional[str] = None, device: int = 0):
        super().__init__()
        if render_mode not in {None, *self.metadata["render_modes"]}:
            raise ValueError(f"Unsupported render mode: {render_mode}")
        self.render_mode = render_mode
        self._vec = ArmSingleVectorEnv(1, final_time, time_step, recording_fps, n_elems, n_action,
                                       control_penalty_coeff, device, autoreset=False)
        self.final_time, self.time_step, self.step_skip = final_time, time_step, self._vec.step_skip
        self.n_elems, self.n_seg, self.n_action = n_elems, n_elems - 1, n_action
        self.action_space = self._vec.single_action_space
        self.observation_space = self._vec.single_observation_space
        self.time = np.float64(0.0)
        self.counter = 0

    def reset(self, *, seed: Optional[int] = None, options: Optional[dict] = None):
        super().reset(seed=seed)
        obs, _ = self._vec.reset()
        self.time = np.float64(0.0)
        self.counter = 0
        return obs[0].cpu().numpy(), {}

    def step(self, action):
        import torch
        a = torch.as_tensor(np.asarray(action, dtype=np.float32).reshape(1, -1), device=self._vec.device)
        obs, reward, term, trunc, _ = self._vec.step(a)
        self.time = _advance_time(self.time, self.time_step, self.step_skip)
        if bool(term[0]) and float(reward[0]) < 0 and not bool((self._vec.prev_dist < 0.1)[0]):
            print(f" Nan detected in, exiting simulation now. {self.time=}")
        timelimit = bool(self.time > self.final_time)
        self.counter += 1
        return (obs[0].cpu().numpy(), np.float64(reward[0].item()), bool(term[0]), timelimit,
                {"time": self.time, "TimeLimit.truncated": timelimit})

    def rod_state(self):
        return {k: v[0].cpu().numpy() for k, v in self._vec.fields().items()}

    def render(self):
        return None

    def close(self):
        self._vec.close()
