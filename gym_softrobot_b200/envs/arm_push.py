"""OctoArmPush-v0 / OctoArmPush-v1 / OctoArmPullWeight-v0 on the B200 kernel.

Host-side mirror of `/root/reference/gym_softrobot/envs/octopus/arm_push_env.py` (`ArmPushEnv`, lines 45-413;
`ArmPullWeightEnv`, lines 516-625): one tapered free arm (n = 40, L = 0.2 m, radius 12 mm -> 1 mm given on the nodes),
`AnalyticalLinearDamper`, a `ControllableFixConstraint` ("sucker") whose index the action moves, and COOMM's
`ApplyMuscles` of which only the transverse muscle is ever activated.  PullWeight adds a rigid cylinder tied to node 0
through `FixedJoint2Rigid` and held upright by `BodyBoundaryCondition`.  The substep loop (lines 287-288) is one
`sr_step` launch; the muscle is evaluated in the kernel every substep (sr_config.tm_*), the sucker index / ratio and
the activation are per-env device arrays written by `set_action`.

COOMM is a third-party package outside the reference tree: its published muscle model is restated (DESIGN.md 2).
`config_early_termination` (arm_push_env.py:309-312,436-452): the episode ends once kinetic + shear + bending energy
drop below 1e-7 J, every reward is -10; the energies are torch reductions over the state with the rod's constants.
"""
from typing import Optional

import numpy as np

from .. import _native as nat
from .fork import ForkableVectorEnv
from ..compat import Box, Discrete, Env
from .soft_pendulum import _advance_time

_ARM = dict(base_length=0.2, base_radius=0.012, tip_radius=0.001, density=700.0, youngs_modulus=1e4,
            shear_modulus=1e4 / 1.5)
_N_ELEM = 40


def arm_push_node_masses(n_elem=_N_ELEM):
    """Nodal masses of the arm as `CosseratRod.straight_rod` builds them from
    `radius_mean = (radius[:-1] + radius[1:]) / 2`, `radius = linspace(base, tip, n + 1)` (arm_push_env.py:161-175)."""
    radius = np.linspace(_ARM["base_radius"], _ARM["tip_radius"], n_elem + 1)
    radius_mean = (radius[:-1] + radius[1:]) / 2
    x = np.linspace(0.0, _ARM["base_length"], n_elem + 1)
    volume = np.pi * radius_mean ** 2 * (x[1:] - x[:-1])
    mass = np.zeros(n_elem + 1)
    mass[:-1] += 0.5 * _ARM["density"] * volume
    mass[1:] += 0.5 * _ARM["density"] * volume
    return mass


def arm_push_energy_tables(n_elem=_N_ELEM):
    """(node mass [n+1], J [3, n], S [3, n], B [3, n-1], rest_lengths [n], rest_voronoi_lengths [n-1]) of the arm, as
    `CosseratRod.straight_rod` allocates them (SURVEY A.1) — what PyElastica's compute_*_energy read."""
    E, G, rho = _ARM["youngs_modulus"], _ARM["shear_modulus"], _ARM["density"]
    radius = np.linspace(_ARM["base_radius"], _ARM["tip_radius"], n_elem + 1)
    radius = (radius[:-1] + radius[1:]) / 2
    x = np.linspace(0.0, _ARM["base_length"], n_elem + 1)
    rl = x[1:] - x[:-1]
    A0 = np.pi * radius * radius
    I1 = A0 * A0 / (4.0 * np.pi)
    I = np.stack([I1, I1, 2.0 * I1])
    J = I * (rho * rl)
    S = np.stack([27.0 / 28.0 * G * A0, 27.0 / 28.0 * G * A0, E * A0])
    Bel = np.stack([E * I[0], E * I[1], G * I[2]])
    B = (Bel[:, 1:] * rl[1:] + Bel[:, :-1] * rl[:-1]) / (rl[1:] + rl[:-1])
    return arm_push_node_masses(n_elem), J, S, B, rl, 0.5 * (rl[1:] + rl[:-1])


def _make_handle(n_env, time_step, device, pull_weight):
    damp = 0.05 * 2 * (5e2 if pull_weight else 1e2)
    kw = {}
    if pull_weight:   # arm_push_env.py:551-586
        kw = dict(n_rod=1, head=dict(length=_ARM["base_radius"] * 2, radius=0.015, density=_ARM["density"] * 1.0),
                  joint=dict(k=1e6, nu=1e-2, kt=1e0, radius=0.015, angles_deg=[0.0]))
    return nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=_N_ELEM, dt=time_step, gravity=(0.0, 0.0, 0.0),
                      damping_constant=damp, bc_kind=nat.BC_FREE, device=device, sucker_index=0, taper_node_mean=True,
                      tm_muscle=dict(max_stress=1.0, radius_ref=_ARM["base_radius"]), **_ARM, **kw)


class ArmPushVectorEnv(ForkableVectorEnv):
    """N independent OctoArmPush / OctoArmPullWeight envs (torch CUDA I/O), one physics launch per env-step.
    `mode` "discrete": actions are an integer tensor [n_env] in {0, 1}; "continuous": float [n_env, 2] in [0, 1]."""

    PER_ENV = ("step_count", "prev_action")   # per-env host state (copy_envs)

    def __init__(self, n_env, final_time=2.5, time_step=5.0e-5, recording_fps=40, mode="discrete",
                 pull_weight=False, device: int = 0, autoreset: bool = True, config_early_termination: bool = False):
        import torch
        self.config_early_termination = config_early_termination
        self.torch = torch
        if mode not in ("discrete", "continuous"):
            raise NotImplementedError(f"The mode {mode} is not available.")
        self.mode = 0 if mode == "discrete" else 1
        self.n_env, self.n_elem, self.pull_weight = n_env, _N_ELEM, pull_weight
        self.final_time, self.time_step = final_time, time_step
        self.step_skip = int(1.0 / (recording_fps * time_step))
        self.device = torch.device(f"cuda:{device}")
        self.autoreset = autoreset
        n_action = 2
        self.single_action_space = Discrete(2) if self.mode == 0 else Box(0.0, 1.0, shape=(n_action,), dtype=np.float32)
        self.single_observation_space = Box(-np.inf, np.inf, shape=((self.n_elem + 1) * 2 + 2,), dtype=np.float32)
        self.handle = _make_handle(n_env, time_step, device, pull_weight)
        self._ratio0 = 0.9 if pull_weight else 1.0       # SuckerController(reduction_ratio=...) of the build
        self._scratch = (torch.empty((n_env, 6), dtype=torch.float32, device=self.device),
                         torch.empty(n_env, dtype=torch.float64, device=self.device),
                         torch.empty(n_env, dtype=torch.uint8, device=self.device))
        m = arm_push_node_masses(self.n_elem)
        self._mass = torch.as_tensor(m, device=self.device)
        self._mass_sum = float(m.sum())
        self._etab = [torch.as_tensor(t, device=self.device) for t in arm_push_energy_tables(self.n_elem)]
        row = [0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0, -0.0]
        if pull_weight:   # the cylinder: start, direction, normal (arm_push_env.py:551-562)
            row += [-0.015 * 0.9, 0.0, -2 * _ARM["base_radius"], 0.0, 0.0, 1.0, 0.0, 1.0, 0.0]
        self._init = np.array([row])
        n_max = int(final_time / (self.step_skip * time_step)) + 8
        table, t = [np.float64(0.0)], np.float64(0.0)
        for _ in range(n_max):
            t = _advance_time(t, time_step, self.step_skip)
            table.append(t)
        self._time_table = np.array(table)
        self._first_truncated = int(np.argmax(self._time_table > final_time))
        self.step_count = torch.zeros(n_env, dtype=torch.int64, device=self.device)
        # (set at construction and by step() only, like the reference: arm_push_env.py:111-113,274)
        self.prev_action = (torch.zeros(n_env, dtype=torch.int64, device=self.device) if self.mode == 0
                            else torch.zeros((n_env, n_action), dtype=torch.float32, device=self.device))

    # -- helpers -----------------------------------------------------------------------------
    def _com(self):
        # compute_position_center_of_mass()[:2]
        x = self.handle.fields()["position_collection"].reshape(self.n_env, 3, self.n_elem + 1)
        return (x[:, :2, :] * self._mass).sum(dim=2) / self._mass_sum

    def desired_hamiltonian(self):
        """cal_desired_Hamiltonian (arm_push_env.py:442-452): translational + rotational + shear + bending energy, with
        PyElastica's expressions; sigma / kappa / dilatation are the stale fields of the last force evaluation, as there."""
        f = self.handle.fields()
        mass, J, S, B, rl, rvl = self._etab
        n = self.n_elem
        v = f["velocity_collection"].reshape(self.n_env, 3, n + 1)
        w = f["omega_collection"].reshape(self.n_env, 3, n)
        sg = f["sigma"].reshape(self.n_env, 3, n)
        kp = f["kappa"].reshape(self.n_env, 3, n - 1)
        e = f["dilatation"].reshape(self.n_env, n)
        trans = 0.5 * (mass * (v * v).sum(dim=1)).sum(dim=1)
        rot = 0.5 * (w * (J * w / e[:, None, :])).sum(dim=1).sum(dim=1)
        shear = 0.5 * ((sg * (S * sg)).sum(dim=1) * rl).sum(dim=1)
        bend = 0.5 * ((kp * (B * kp)).sum(dim=1) * rvl).sum(dim=1)
        return trans + rot + shear + bend

    def _obs(self):
        torch = self.torch
        f = self.handle.fields()
        pos = f["position_collection"].reshape(self.n_env, 3, self.n_elem + 1)[:, 0, :]
        vel = f["velocity_collection"].reshape(self.n_env, 3, self.n_elem + 1)[:, 0, :]
        if self.mode == 0:
            tail = torch.nn.functional.one_hot(self.prev_action, 2).double()     # np.eye(2)[previous_action]
        else:
            tail = self.prev_action.double()
        return torch.cat([pos, vel, tail], dim=1).float()

    def _reset_envs(self, idx=None):
        torch = self.torch
        n = self.n_env if idx is None else int(idx.numel())
        init = torch.as_tensor(np.repeat(self._init, n, axis=0), device=self.device).contiguous()
        self.handle.reset(init, None if idx is None else idx.to(torch.int32).contiguous())
        sel = slice(None) if idx is None else idx
        # a fresh build: SuckerController(index=0, reduction_ratio) turned on, muscles at rest
        self.handle.sucker_tensor()[sel] = self._ratio0
        self.handle.sucker_index_tensor()[sel] = 0
        self.handle.tm_activation_tensor()[sel] = 0.0

    def reset(self, seed: int = 0):
        self._reset_envs()
        self.step_count.zero_()
        return self._obs(), {}

    def set_action(self, action):
        torch = self.torch
        idx_t, act_t = self.handle.sucker_index_tensor(), self.handle.tm_activation_tensor()
        if self.mode == 0:
            a = action.to(device=self.device, dtype=torch.int64).reshape(self.n_env)
            if bool(((a != 0) & (a != 1)).any()):
                raise NotImplementedError("Action must be 1 or 0")
            # 0: hold node 0 and contract the transverse muscle; 1: hold the last node and release
            idx_t[:] = torch.where(a == 0, 0, -1).to(torch.int32)
            act_t[:] = torch.where(a == 0, 0.5, 0.0).double()
            self.prev_action = a.clone()
        else:
            a = action.to(device=self.device, dtype=torch.float32).reshape(self.n_env, 2)
            # int(np.clip(location * n_elem, 0, n_elem - 1)) on the float32 action
            idx_t[:] = torch.clamp(a[:, 0] * self.n_elem, 0, self.n_elem - 1).to(torch.int32)
            act_t[:] = a[:, 1].double()
            self.prev_action = a.clone()

    def step(self, action):
        torch = self.torch
        self.set_action(action)
        prev_cm = self._com()
        obs6, rew, term = self._scratch
        self.handle.step(None, self.step_skip, obs6, rew, term)
        self.step_count += 1
        cm = self._com()
        f = self.handle.fields()
        invalid = term.bool()
        for k in ("director_collection", "omega_collection"):
            invalid = invalid | torch.isnan(f[k].reshape(self.n_env, -1)).any(dim=1)
        invalid = invalid | torch.isnan(cm).any(dim=1)
        forward = cm.norm(dim=1) - prev_cm.norm(dim=1)
        reward = torch.where(invalid, torch.full_like(forward, -20.0), forward)
        terminated = invalid.clone()
        truncated = self.step_count >= self._first_truncated
        if self.config_early_termination:
            # arm_push_env.py:309-312: this branch comes first — no NaN penalty, no forward reward, always -10
            terminated = self.desired_hamiltonian() < 1e-7
            truncated = truncated | terminated
            reward = torch.full_like(forward, -10.0)
        bad = torch.isnan(reward)
        terminated |= bad
        reward = torch.where(bad, torch.full_like(reward, -20.0), reward)
        obs = self._obs()
        bad = torch.isnan(obs).any(dim=1)
        terminated |= bad
        reward = torch.where(bad, torch.full_like(reward, -20.0), reward)
        obs = torch.nan_to_num(obs)
        info = {"time": torch.as_tensor(self._time_table, device=self.device)[
            self.step_count.clamp(max=len(self._time_table) - 1)]}
        info["TimeLimit.truncated"] = truncated.clone()
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


class ArmPushEnv(Env):
    """Drop-in for the reference `ArmPushEnv` (same kwargs; arm_push_env.py:65-74): a batch of one."""

    metadata = {"render_modes": ["rgb_array", "human"], "render_fps": 40}
    _pull_weight = False

    def __init__(self, final_time: float = 2.5, time_step: float = 5.0e-5, recording_fps: int = 40,
                 mode: str = "discrete", config_generate_video: bool = False, config_early_termination: bool = False,
                 render_mode: Optional[str] = None, device: int = 0):
        super().__init__()
        if render_mode not in {None, *self.metadata["render_modes"]}:
            raise ValueError(f"Unsupported render mode: {render_mode}")
        self.render_mode = render_mode
        self._vec = ArmPushVectorEnv(1, final_time, time_step, recording_fps, mode, self._pull_weight, device,
                                     autoreset=False, config_early_termination=config_early_termination)
        self.final_time, self.time_step, self.step_skip = final_time, time_step, self._vec.step_skip
        self.total_steps = int(final_time / time_step)
        self.recording_fps, self.n_elem, self.mode = recording_fps, _N_ELEM, self._vec.mode
        self.action_space = self._vec.single_action_space
        self.observation_space = self._vec.single_observation_space
        self.config_generate_video, self.config_early_termination = config_generate_video, config_early_termination
        self.time = np.float64(0.0)

    def reset(self, *, seed: Optional[int] = None, options: Optional[dict] = None):
        super().reset(seed=seed)
        obs, _ = self._vec.reset()
        self.time = np.float64(0.0)
        return obs[0].cpu().numpy(), {}

    def step(self, action):
        import torch
        if self.mode == 0:
            a = torch.as_tensor(np.asarray(action, dtype=np.int64).reshape(1), device=self._vec.device)
        else:
            a = torch.as_tensor(np.asarray(action, dtype=np.float32).reshape(1, -1), device=self._vec.device)
        obs, reward, term, trunc, _ = self._vec.step(a)
        self.time = _advance_time(self.time, self.time_step, self.step_skip)
        timelimit = bool(self.time > self.final_time)
        # (with config_early_termination the reference sets truncated = terminated first, then the time limit ORs in)
        truncated = timelimit or (self.config_early_termination and bool(term[0]))
        return (obs[0].cpu().numpy(), np.float64(reward[0].item()), bool(term[0]), truncated,
                {"time": self.time, "TimeLimit.truncated": timelimit})

    def check_early_termination(self, cutoff_error=1e-7):
        return bool(self.cal_desired_Hamiltonian() < cutoff_error)

    def cal_desired_Hamiltonian(self):
        return float(self._vec.desired_hamiltonian()[0].item())

    def rod_state(self):
        return {k: v[0].cpu().numpy() for k, v in self._vec.fields().items()}

    def head_state(self):
        return self._vec.handle.head_tensor()[0].cpu().numpy()

    def render(self):
        return None

    def close(self):
        self._vec.close()


class ArmPullWeightEnv(ArmPushEnv):
    """Drop-in for the reference `ArmPullWeightEnv` (arm_push_env.py:516-625): time_step 2.5e-5, the arm drags a
    rigid cylinder."""

    _pull_weight = True

    def __init__(self, **kwargs):
        super().__init__(time_step=2.5e-5, **kwargs)
