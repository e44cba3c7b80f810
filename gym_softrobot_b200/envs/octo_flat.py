"""OctoFlat-v0 / OctoFlatLite-v0 on the B200 kernel.

Host-side mirror of `/root/reference/gym_softrobot/envs/octopus/flat_env.py` (`FlatEnv`, lines 41-408)
and `build_octopus` (`envs/octopus/build.py:52-217`): `n_arm` arms around a rigid Cylinder head held
upright by `BodyBoundaryCondition`, tied to it by `FixedJoint2Rigid` joints, lying on a frictional plane,
actuated through the arms' rest curvature (cubic interpolation of `n_action` control values padded with
zeros at both ends, lines 288-311).  One `sr_step` launch advances every arm and head of every env by
`step_skip` substeps; observation / reward are small torch reductions in the reference's order.
"""
from typing import Optional

import numpy as np

from .. import _native as nat
from .fork import ForkableVectorEnv
from ..compat import Box, Dict, Env
from .arm_single import arm_contact_params, _ROD, _G
from .soft_pendulum import _advance_time

_HEAD_RADIUS, _HEAD_DENSITY = 0.04, 700.0     # build.py:39-40
_JOINT = dict(k=1e6, nu=1e-3, kt=1e0)          # build.py:37-38,126-128


def octopus_init_params(n_arm):
    """start/direction/normal of every arm + of the head cylinder (build.py:66-106), one row."""
    from scipy.spatial.transform import Rotation as Rot
    r0 = _ROD["base_radius"]
    row = []
    for arm_i in range(n_arm):
        rot = Rot.from_euler("z", 360 / n_arm * arm_i, degrees=True)
        row += list(rot.apply([_HEAD_RADIUS, 0.0, 0.0])) + list(rot.apply([1.0, 0.0, 0.0])) + [0.0, 0.0, 1.0]
    row += [0.0, 0.0, -r0] + [0.0, 0.0, 1.0] + [0.0, 1.0, 0.0]
    return np.array([row], dtype=np.float64)


def padded_curvature_interp_matrix(n_action, n_seg):
    """flat_env.py:296-309: zero-pad the control values at both ends, cubic-interpolate to n_seg points;
    linear in the action, so a fixed [n_seg, n_action] matrix (built with scipy once)."""
    from scipy.interpolate import interp1d
    xs, xq = np.linspace(0, 1, n_action + 2), np.linspace(0, 1, n_seg)
    cols = []
    for i in range(n_action):
        a = np.zeros(n_action + 2); a[i + 1] = 1.0
        cols.append(interp1d(xs, a, kind="cubic", axis=-1)(xq))
    return np.stack(cols, axis=1)


def count_crossings(p1, p2):
    """Number of intersections of two planar polylines per env (`utils/intersection.py:30-77`):
    segment pairs whose bounding boxes overlap and whose line parameters both lie in [0, 1].
    p1, p2: [N, 2, m] tensors."""
    import torch
    a0, a1 = p1[:, :, :-1].unsqueeze(3), p1[:, :, 1:].unsqueeze(3)      # [N,2,m-1,1]
    b0, b1 = p2[:, :, :-1].unsqueeze(2), p2[:, :, 1:].unsqueeze(2)      # [N,2,1,m-1]
    box = ((torch.minimum(a0, a1) <= torch.maximum(b0, b1)) & (torch.maximum(a0, a1) >= torch.minimum(b0, b1))).all(dim=1)
    da, db, dab = a1 - a0, b1 - b0, b0 - a0
    den = da[:, 0] * db[:, 1] - da[:, 1] * db[:, 0]
    t1 = (dab[:, 0] * db[:, 1] - dab[:, 1] * db[:, 0]) / den
    t2 = (dab[:, 0] * da[:, 1] - dab[:, 1] * da[:, 0]) / den
    hit = box & (t1 >= 0) & (t1 <= 1) & (t2 >= 0) & (t2 <= 1)
    return hit.sum(dim=(1, 2))


class OctoFlatVectorEnv(ForkableVectorEnv):
    """N independent OctoFlat-v0 envs, torch CUDA I/O.  `policy_mode` as in the reference (flat_env.py:84-145,
    248-271): "decentralized" declares a per-arm action space and appends the arm's one-hot id to each
    row of the individual observation; the physics and the batched action layout are the same."""

    PER_ENV = ("step_count", "prev_action", "target")   # per-env host state (copy_envs)

    def __init__(self, n_env, final_time=5.0, time_step=7.0e-5, recording_fps=5, n_elems=10, n_arm=8,
                 n_action=3, device: int = 0, autoreset: bool = True, env_offset: int = 0,
                 policy_mode: str = "centralized"):
        import torch
        self.torch = torch
        self.n_env, self.n_elems, self.n_seg, self.n_arm, self.n_action = n_env, n_elems, n_elems - 1, n_arm, n_action
        self.final_time, self.time_step = final_time, time_step
        self.step_skip = int(1.0 / (recording_fps * time_step))
        self.device = torch.device(f"cuda:{device}")
        self.autoreset, self.env_offset = autoreset, env_offset
        if policy_mode not in ("centralized", "decentralized"):
            raise NotImplementedError(policy_mode)
        self.policy_mode = policy_mode
        d_ind = self.n_seg + (n_elems + 1) * 4 + n_action
        if policy_mode == "centralized":
            lo = np.repeat(np.ones(n_action) * -22, n_arm)
            self.single_action_space = Box(lo, -lo, shape=(n_arm * n_action,), dtype=np.float32)
            self.obs_shapes = {"individual": (n_arm, d_ind), "shared": (13,)}
        else:
            lo = np.ones(n_action) * -22
            self.single_action_space = Box(lo, -lo, shape=(n_action,), dtype=np.float32)
            self.obs_shapes = {"individual": (d_ind + n_arm,), "shared": (13,)}
        r0 = _ROD["base_radius"]
        self.handle = nat.Handle(
            model=nat.MODEL_ROD, n_env=n_env, n_elem=n_elems, dt=time_step, gravity=(0.0, 0.0, _G),
            damping_constant=1e-2, bc_kind=nat.BC_FREE, device=device, contact=arm_contact_params(), n_rod=n_arm,
            head=dict(length=r0 * 2, radius=_HEAD_RADIUS, density=_HEAD_DENSITY),
            joint=dict(radius=_HEAD_RADIUS, angles_deg=[360 / n_arm * a for a in range(n_arm)], **_JOINT), **_ROD)
        self._W = torch.as_tensor(padded_curvature_interp_matrix(n_action, self.n_seg), device=self.device)
        self._init_row = octopus_init_params(n_arm)
        self._scratch = (torch.empty((n_env, 6), dtype=torch.float32, device=self.device),
                         torch.empty(n_env, dtype=torch.float64, device=self.device),
                         torch.empty(n_env, dtype=torch.uint8, device=self.device))
        n_max = int(final_time / (self.step_skip * time_step)) + 8
        table, t = [np.float64(0.0)], np.float64(0.0)
        for _ in range(n_max):
            t = _advance_time(t, time_step, self.step_skip)
            table.append(t)
        self._time_table = np.array(table)
        self._first_truncated = int(np.argmax(self._time_table > final_time))
        self.step_count = torch.zeros(n_env, dtype=torch.int64, device=self.device)
        self.prev_action = torch.zeros((n_env, n_arm * n_action), dtype=torch.float32, device=self.device)
        self.target = torch.zeros((n_env, 2), dtype=torch.float64, device=self.device)
        self._seed, self._n_autoreset = 0, 0

    def _targets(self, env_ids, initial):
        # flat_env.py:223: (2 - 0.5) * np_random.random(2) + 0.5.  reset(seed): env i draws like a reference
        # env reset with seed + global index; autoreset: one batched stream
        if initial:
            u = np.array([np.random.Generator(np.random.PCG64(np.random.SeedSequence(
                int(self._seed + self.env_offset + i)))).random(2) for i in env_ids])
        else:
            self._n_autoreset += 1
            ss = np.random.SeedSequence([int(self._seed), int(self.env_offset), int(self._n_autoreset)])
            u = np.random.Generator(np.random.PCG64(ss)).random((len(env_ids), 2))
        return (2 - 0.5) * u + 0.5

    def _fields(self):
        """Rod views with an explicit arm axis, [n_env, n_arm, ...], also for the single-arm Lite env."""
        f = self.handle.fields()
        return f if self.n_arm > 1 else {k: v.unsqueeze(1) for k, v in f.items()}

    def _obs(self):
        torch = self.torch
        f, hd = self._fields(), self.handle.head_tensor()
        c = hd[:, None, 0:2, None]                                   # head centre (x, y)
        x, v = f["position_collection"], f["velocity_collection"]
        pa = self.prev_action.reshape(self.n_env, self.n_arm, self.n_action).double()
        cols = [f["kappa"][:, :, 0, :], x[:, :, 0, :] - c[:, :, 0], x[:, :, 1, :] - c[:, :, 1],
                v[:, :, 0, :], v[:, :, 1, :], pa]
        if self.policy_mode == "decentralized":
            cols.append(torch.eye(self.n_arm, dtype=torch.float64, device=self.device).expand(self.n_env, -1, -1))
        ind = torch.cat(cols, dim=2).float()
        shared = torch.cat([self.target - hd[:, 0:2], hd[:, 3:5], hd[:, 6:15]], dim=1).float()
        return {"individual": ind, "shared": shared}

    def _reset_envs(self, idx=None, initial=False):
        torch = self.torch
        ids = np.arange(self.n_env) if idx is None else idx.cpu().numpy()
        init = torch.as_tensor(np.repeat(self._init_row, len(ids), axis=0), device=self.device).contiguous()
        self.handle.reset(init, None if idx is None else idx.to(torch.int32).contiguous())
        rk = self.handle.rest_kappa_tensor().unflatten(0, (self.n_env, self.n_arm))
        if idx is None:
            rk.zero_()
        else:
            rk[idx] = 0
        self.target[ids] = torch.as_tensor(self._targets(ids, initial), device=self.device)

    def reset(self, seed: int = 0):
        self._seed = seed
        self._n_autoreset = 0
        self._reset_envs(initial=True)
        self.step_count.zero_()
        # (the previous action survives a reset, as in the reference: flat_env.py:135-139,288-293)
        return self._obs(), {}

    def step(self, action):
        torch = self.torch
        action = action.to(device=self.device, dtype=torch.float32).reshape(self.n_env, self.n_arm * self.n_action)
        self.prev_action = action.clone()
        # rest curvature = W a, accumulated control point by control point (fixed order: a GEMM would
        # pick batch-size dependent kernels and make results depend on n_env at the 1e-16 level)
        a3 = action.double().reshape(self.n_env, self.n_arm, self.n_action)
        kap = a3[:, :, 0:1] * self._W[:, 0]
        for k in range(1, self.n_action):
            kap = kap + a3[:, :, k:k + 1] * self._W[:, k]                                 # [N, arm, n_seg]
        self.handle.rest_kappa_tensor().unflatten(0, (self.n_env, self.n_arm))[:, :, 0, :] = kap
        hd = self.handle.head_tensor()
        xposbefore = hd[:, 0:2].clone()
        o6, rew, term = self._scratch
        self.handle.step(None, self.step_skip, o6, rew, term)
        self.step_count += 1
        invalid = term.bool()
        xy = self._fields()["position_collection"][:, :, :2, :]                  # [N, arm, 2, n+1]
        crossing = torch.zeros(self.n_env, dtype=torch.int64, device=self.device)
        for i in range(self.n_arm - 1):                                          # pairs (i-1, i), as the reference
            crossing += count_crossings(xy[:, i - 1], xy[:, i])
        dist = (self.target - hd[:, 0:2]).norm(dim=1)
        forward = (dist - (self.target - xposbefore).norm(dim=1)) / (self.step_skip * self.time_step)
        touched = (dist < 0.1) & ~invalid
        survive = torch.where(invalid, torch.full_like(dist, -50.0),
                              torch.where(touched, torch.full_like(dist, 100.0), -0.02 * crossing.double()))
        reward = torch.where(invalid, torch.zeros_like(dist), forward) + survive
        terminated = invalid | touched
        reward = torch.where(terminated, reward - (dist - 0.1), reward)
        truncated = self.step_count >= self._first_truncated
        obs = self._obs()
        info = {"time": torch.as_tensor(self._time_table, device=self.device)[
            self.step_count.clamp(max=len(self._time_table) - 1)], "arm_crossing": crossing}
        done = terminated | truncated
        if self.autoreset and bool(done.any()):
            idx = torch.nonzero(done).flatten()
            info["final_obs"] = {k: v[idx].clone() for k, v in obs.items()}
            info["reset_idx"] = idx
            self._reset_envs(idx)
            self.step_count[idx] = 0
            fresh = self._obs()
            for k in obs:
                obs[k][idx] = fresh[k][idx]
        return obs, reward, terminated, truncated, info

    def fields(self):
        return self._fields()

    def close(self):
        self.handle.close()


class FlatEnv(Env):
    """Drop-in for the reference `FlatEnv` (flat_env.py:54-66, both policy modes): a batch of one."""

    metadata = {"render_modes": ["rgb_array", "human"], "render_fps": 5}

    def __init__(self, final_time=5.0, time_step=7.0e-5, recording_fps=5, n_elems=10, n_arm=8, n_action=3,
                 config_generate_video=False, config_save_head_data=False, policy_mode="centralized",
                 render_mode: Optional[str] = None, device: int = 0):
        super().__init__()
        if render_mode not in {None, *self.metadata["render_modes"]}:
            raise ValueError(f"Unsupported render mode: {render_mode}")
        self.render_mode = render_mode
        self.policy_mode = policy_mode
        self._vec = OctoFlatVectorEnv(1, final_time, time_step, recording_fps, n_elems, n_arm, n_action, device,
                                      autoreset=False, policy_mode=policy_mode)
        self.final_time, self.time_step, self.step_skip = final_time, time_step, self._vec.step_skip
        self.n_arm, self.n_elems, self.n_action = n_arm, n_elems, n_action
        self.action_space = self._vec.single_action_space
        # flat_env.py:99-130: the declared individual shape is per arm in decentralized mode
        shapes = self._vec.obs_shapes
        self.observation_space = Dict({
            "individual": Box(-np.inf, np.inf, shape=shapes["individual"], dtype=np.float32),
            "shared": Box(-np.inf, np.inf, shape=shapes["shared"], dtype=np.float32)})
        self.time = np.float64(0.0)
        self.counter = 0

    def reset(self, *, seed: Optional[int] = None, options: Optional[dict] = None):
        super().reset(seed=seed)
        self._vec._reset_envs()
        # the target comes from the env's own generator, exactly like flat_env.py:223
        import torch
        self._target = (2 - 0.5) * self.np_random.random(2) + 0.5
        self._vec.target[0] = torch.as_tensor(self._target, device=self._vec.device)
        self._vec.step_count.zero_()
        self.time = np.float64(0.0)
        self.counter = 0
        return {k: v[0].cpu().numpy() for k, v in self._vec._obs().items()}, {}

    def step(self, action):
        import torch
        a = torch.as_tensor(np.asarray(action, dtype=np.float32).reshape(1, -1), device=self._vec.device)
        obs, reward, term, trunc, _ = self._vec.step(a)
        self.time = _advance_time(self.time, self.time_step, self.step_skip)
        timelimit = bool(self.time > self.final_time)
        self.counter += 1
        return ({k: v[0].cpu().numpy() for k, v in obs.items()}, float(reward[0].item()), bool(term[0]), timelimit,
                {"time": self.time, "TimeLimit.truncated": timelimit})

    def state(self):
        f = {k: v[0].cpu().numpy() for k, v in self._vec.fields().items()}
        f["head"] = self._vec.handle.head_tensor()[0].cpu().numpy()
        return f

    def render(self):
        return None

    def close(self):
        self._vec.close()
