"""OctoArmTwo-v0 on the B200 kernel.

Host-side mirror of `/root/reference/gym_softrobot/envs/octopus/arm_two_env.py` (`ArmTwoEnv`, lines 37-347) over
`build_two_arms` (`envs/octopus/build_muscle_octopus.py:182-291`): two tapered arms at 90 / 270 degrees on a light
rigid head (`FixedJoint2Rigid`, `BodyBoundaryCondition`), three `ControllableFixConstraint`s ("suckers") per arm at fixed
elements, and COOMM's `ApplyMuscles` with all three muscle layers.  Per arm the action is (3 sucker ratios, 3
longitudinal control values, 3 transverse control values); the control values become per-element activations through a
cubic `interp1d` over (0, sucker locations, n_elems - 1) (arm_two_env.py:236-247) — linear in the values, so one small
matrix product here.  The substep loop (arm_two_env.py:262-263) is one `sr_step` launch of the muscle-layer kernel.

COOMM is a third-party package outside the reference tree: its published muscle model is restated (DESIGN.md 2).
"""
from typing import Optional

import numpy as np

from .. import _native as nat
from .fork import ForkableVectorEnv
from ..compat import Box, Env
from .octo_crawl import _ARM, _DAMPER_TIME_STEP, _HEAD_DENSITY, _HEAD_RADIUS, _JOINT
from .octo_reach import _LM_MAX_STRESS, _TM_MAX_STRESS, es_longitudinal_positions
from .soft_pendulum import _advance_time

_N_ARM, _N_SUCKER = 2, 3


def two_arm_init_params():
    """[9 * (2 + 1)] start / direction / normal of the two arms, then of the head cylinder
    (build_muscle_octopus.py:199-224)."""
    angles = [90.0 + 180.0 * i for i in range(_N_ARM)]
    row = []
    for ang in angles:
        c, s = np.cos(np.deg2rad(ang)), np.sin(np.deg2rad(ang))
        row += [c * _HEAD_RADIUS, s * _HEAD_RADIUS, 0.0, c, s, 0.0, 0.0, 0.0, 1.0]
    row += [0.0, 0.0, -_ARM["base_radius"] * 2, 0.0, 0.0, 1.0, 0.0, 1.0, 0.0]
    return np.array([row]), angles


def activation_interp_matrix(control_location, n_elems):
    """`interp1d(control_location, [0] + list(a) + [0], kind="cubic")(range(n_elems))` is linear in `a`: [n_elems, 3]."""
    from scipy.interpolate import interp1d
    cols = []
    for i in range(_N_SUCKER):
        y = np.zeros(len(control_location))
        y[1 + i] = 1.0
        cols.append(interp1d(control_location, y, kind="cubic")(range(n_elems)))
    return np.stack(cols, axis=1)


class ArmTwoVectorEnv(ForkableVectorEnv):
    """N independent OctoArmTwo-v0 envs (torch CUDA I/O), one physics launch per env-step; actions float [n_env, 18]."""

    PER_ENV = ("step_count", "prev_action", "prev_kappa")   # per-env host state (copy_envs)

    def __init__(self, n_env, final_time=5.0, time_step=5.0e-5, recording_fps=25, n_elems=20, device: int = 0,
                 autoreset: bool = True):
        import torch
        self.torch = torch
        self.n_env, self.n_arm, self.n_elems, self.n_seg, self.n_action = n_env, _N_ARM, n_elems, n_elems - 1, 9
        self.n_sucker = _N_SUCKER
        self.sucker_location = [n_elems // (_N_SUCKER * 2) * (2 * i + 1) for i in range(_N_SUCKER)]
        self.control_location = [0] + self.sucker_location + [n_elems - 1]
        self.final_time, self.time_step = final_time, time_step
        self.step_skip = int(1.0 / (recording_fps * time_step))
        self.device = torch.device(f"cuda:{device}")
        self.autoreset = autoreset
        self.shared_space = 3
        obs_dim = self.n_arm * (self.n_seg * 2 + self.n_action + self.n_arm + self.shared_space)
        self.single_action_space = Box(0.0, 1.0, shape=(self.n_arm * self.n_action,), dtype=np.float32)
        self.single_observation_space = Box(-np.inf, np.inf, shape=(obs_dim,), dtype=np.float32)
        self._init, angles = two_arm_init_params()
        damp = 0.20 * 1e-2 * (_DAMPER_TIME_STEP / time_step)     # (see octo_crawl.py: the damper's literal time step)
        self.handle = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n_elems, dt=time_step, gravity=(0.0, 0.0, 0.0),
                                 damping_constant=damp, bc_kind=nat.BC_FREE, device=device, n_rod=self.n_arm,
                                 head=dict(length=_ARM["base_radius"] * 2, radius=_HEAD_RADIUS, density=_HEAD_DENSITY),
                                 joint=dict(radius=_HEAD_RADIUS, angles_deg=angles, **_JOINT),
                                 tm_muscle=dict(max_stress=_TM_MAX_STRESS, radius_ref=_ARM["base_radius"]),
                                 muscle_layers=dict(lm_max_stress=_LM_MAX_STRESS, lm_positions=es_longitudinal_positions()),
                                 fixed_suckers=self.sucker_location, **_ARM)
        self._W = torch.as_tensor(activation_interp_matrix(self.control_location, n_elems), device=self.device)   # [n, 3] f64
        self._scratch = (torch.empty((n_env, 6), dtype=torch.float32, device=self.device),
                         torch.empty(n_env, dtype=torch.float64, device=self.device),
                         torch.empty(n_env, dtype=torch.uint8, device=self.device))
        self._target = torch.tensor([5.0, 0.0], dtype=torch.float64, device=self.device)
        self._eye = torch.eye(self.n_arm, dtype=torch.float64, device=self.device)
        n_max = int(final_time / (self.step_skip * time_step)) + 8
        table, t = [np.float64(0.0)], np.float64(0.0)
        for _ in range(n_max):
            t = _advance_time(t, time_step, self.step_skip)
            table.append(t)
        self._time_table = torch.as_tensor(np.array(table), device=self.device)
        self.step_count = torch.zeros(n_env, dtype=torch.int64, device=self.device)
        # (set at construction and by set_action / get_state only, like the reference: arm_two_env.py:103-106,220,248)
        self.prev_action = torch.zeros((n_env, self.n_arm, self.n_action), dtype=torch.float32, device=self.device)
        self.prev_kappa = torch.zeros((n_env, self.n_arm, self.n_seg), dtype=torch.float32, device=self.device)

    # -- helpers -----------------------------------------------------------------------------
    def _head_xy(self):
        return self.handle.head_tensor()[:, 0:2]

    def _obs(self, sel=None):
        """get_state (arm_two_env.py:186-220); refreshes prev_kappa of the envs in `sel` (all when None) like the
        reference's get_state does on every call."""
        torch = self.torch
        f = self.handle.fields()
        N, A = self.n_env, self.n_arm
        kappa = f["kappa"][:, :, 0, :]
        hd = self.handle.head_tensor()
        shared = hd[:, 3:6].float().double()
        obs = torch.cat([kappa, self.prev_kappa.double(), self.prev_action.double(), self._eye.expand(N, A, A),
                         shared[:, None, :].expand(N, A, self.shared_space)], dim=2)
        if sel is None:
            self.prev_kappa = kappa.float()
        else:
            self.prev_kappa[sel] = kappa[sel].float()
        return torch.nan_to_num(obs.float().reshape(N, -1))

    def _reset_envs(self, idx=None):
        torch = self.torch
        n = self.n_env if idx is None else int(idx.numel())
        init = torch.as_tensor(np.repeat(self._init, n, axis=0), device=self.device).contiguous()
        self.handle.reset(init, None if idx is None else idx.to(torch.int32).contiguous())
        sel = slice(None) if idx is None else idx
        view = lambda t: t.unflatten(0, (self.n_env, self.n_arm))
        # a fresh build: SuckerController(reduction_ratio 1.0) turned on (arm_two_env.py:133-152), muscles at rest
        view(self.handle.fixed_sucker_tensor())[sel] = 1.0
        view(self.handle.muscle_activation_tensor())[sel] = 0.0

    def reset(self, seed: Optional[int] = None):
        self._reset_envs()
        self.step_count.zero_()
        return self._obs(), {}

    def muscle_activations(self, action):
        """[n_env, n_arm, 3, n_elems] float64 activations of (LM1, LM2, TM) from a float32 action (arm_two_env.py:236-247)."""
        torch = self.torch
        a = action.to(device=self.device, dtype=torch.float32).reshape(self.n_env, self.n_arm, self.n_action)
        lm = a[:, :, 3:6] - 0.5                                   # float32 arithmetic, as numpy does on the float32 action
        lm1 = torch.clamp(lm, min=0.0).double()
        lm2 = torch.clamp(lm, max=0.0).abs().double()
        tm = a[:, :, 6:9].double()
        ctrl = torch.stack([lm1, lm2, tm], dim=2)                 # [N, A, 3 muscles, 3 control values]
        return ctrl @ self._W.T                                   # [N, A, 3, n_elems]

    def set_action(self, action):
        torch = self.torch
        a = action.to(device=self.device, dtype=torch.float32).reshape(self.n_env, self.n_arm, self.n_action)
        self.handle.fixed_sucker_tensor()[:] = a[:, :, 0:3].double().reshape(-1, 3)
        self.handle.muscle_activation_tensor()[:] = self.muscle_activations(a).reshape(-1, 3, self.n_elems)
        self.prev_action = a.clone()

    def step(self, action):
        torch = self.torch
        self.set_action(action)
        before = self._head_xy().clone()
        obs6, rew, term = self._scratch
        self.handle.step(None, self.step_skip, obs6, rew, term)
        self.step_count += 1
        obs = self._obs()
        invalid = term.bool()        # NaN in any arm's position / velocity
        after = self._head_xy()
        d_after = (self._target - after).norm(dim=1)
        forward = ((self._target - before).norm(dim=1) - d_after) * 1e2
        reached = (d_after < 0.2) & ~invalid
        terminated = invalid | reached
        time = self._time_table[self.step_count.clamp(max=self._time_table.numel() - 1)]
        truncated = ~terminated & (time > self.final_time)
        forward = torch.where(truncated, forward - d_after, forward)
        reward = torch.where(invalid, torch.full_like(forward, -5.0), forward + torch.where(reached, 5.0, 0.0))
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
            obs[idx] = self._obs(idx)[idx]
        return obs, reward, terminated, truncated, info

    def fields(self):
        return self.handle.fields()

    def close(self):
        self.handle.close()


class ArmTwoEnv(Env):
    """Drop-in for the reference `ArmTwoEnv` (same kwargs; arm_two_env.py:56-63): a batch of one."""

    metadata = {"render_modes": ["rgb_array"], "render_fps": 25}

    def __init__(self, final_time=5.0, time_step=5.0e-5, recording_fps=25, n_elems=20,
                 render_mode: Optional[str] = None, device: int = 0):
        super().__init__()
        if render_mode not in {None, *self.metadata["render_modes"]}:
            raise ValueError(f"Unsupported render mode: {render_mode}")
        self.render_mode = render_mode
        self._vec = ArmTwoVectorEnv(1, final_time, time_step, recording_fps, n_elems, device, autoreset=False)
        self.final_time, self.time_step, self.recording_fps = final_time, time_step, recording_fps
        self.total_steps = int(final_time / time_step)
        self.step_skip = self._vec.step_skip
        self.n_arm, self.n_sucker = _N_ARM, _N_SUCKER
        self.n_elems, self.n_seg, self.n_action = n_elems, n_elems - 1, 9
        self.sucker_location, self.control_location = self._vec.sucker_location, self._vec.control_location
        self.grid_size, self.reward_range = 1, 100.0
        self.action_space = self._vec.single_action_space
        self.observation_space = self._vec.single_observation_space
        self.time = np.float64(0.0)
        self.counter = 0
        self._target = np.array([5, 0], dtype=np.float32)

    def get_env_info(self):
        return dict(n_actions=self.n_action, n_agents=8)     # (sic: arm_two_env.py:114-115)

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
        self.counter += 1
        return obs[0].cpu().numpy(), float(reward[0].item()), bool(term[0]), bool(trunc[0]), {"time": self.time}

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
