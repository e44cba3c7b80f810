"""Forking envs (sr_copy_envs, Handle.copy_envs, the vector envs' copy_envs): a destination env takes everything that
evolves or parametrises its source and then continues bit for bit like it, for every model the library steps.

CPU: the index checks and the argument checks ahead of any CUDA call.  GPU: per model, seven envs with different
histories are forked within the handle (a fan-out, then a swap) and compared row by row with a twin handle that ran
the same histories without a copy; copies between handles; every vector env."""

import numpy as np
import pytest

from gym_softrobot_b200 import _native as nat

N_ENV = 7
FORK = ([4, 5, 6, 0], [1, 1, 2, 3])   # (dst, src): a fan-out of env 1, then 2 and 3 over other envs
SWAP = ([1, 2], [2, 1])
# after both copies env e holds the history of env SOURCE_OF[e] of the twin; env 3 was never a destination
SOURCE_OF = [3, 2, 1, 3, 1, 1, 2]


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_copy_env_indices_accepts_ints_sequences_arrays_and_tensors():
    import torch
    d, s = nat.copy_env_indices(3, 0, 4, 1)
    assert d.tolist() == [3] and s.tolist() == [0] and d.dtype == np.int64
    d, s = nat.copy_env_indices(range(4), [0] * 4, 4, 1)
    assert d.tolist() == [0, 1, 2, 3] and s.tolist() == [0, 0, 0, 0]
    d, s = nat.copy_env_indices(np.array([2, 0], np.int32), torch.tensor([1, 1]), 3, 2)
    assert d.tolist() == [2, 0] and s.tolist() == [1, 1]
    d, s = nat.copy_env_indices([], [], 3, 3)
    assert d.size == 0 and s.size == 0
    d, s = nat.copy_env_indices([0, 1], [1, 0], 2, 2)      # a swap: sources may be destinations too
    assert d.tolist() == [0, 1] and s.tolist() == [1, 0]


@pytest.mark.parametrize("dst,src,n_dst,n_src,msg", [
    ([0, 1], [0], 4, 4, "differ in length"),
    ([4], [0], 4, 4, "dst_idx out of range"),
    ([-1], [0], 4, 4, "dst_idx out of range"),
    ([0], [1], 4, 1, "src_idx out of range"),
    ([0], [-2], 4, 4, "src_idx out of range"),
    ([1, 2, 1], [0, 0, 0], 4, 4, "twice"),
    ([0.0], [1], 4, 4, "integers"),
    (np.array([0.5]), np.array([1]), 4, 4, "integers"),
    ([True], [0], 4, 4, "integers"),
    ([[0, 1]], [[1, 0]], 4, 4, "one-dimensional"),
], ids=["lengths", "dst-high", "dst-negative", "src-high", "src-negative", "duplicate", "float-list", "float-array",
        "bool", "2d"])
def test_copy_env_indices_rejects(dst, src, n_dst, n_src, msg):
    with pytest.raises(ValueError, match=msg):
        nat.copy_env_indices(dst, src, n_dst, n_src)


def test_copy_env_indices_rejects_float_tensors():
    import torch
    with pytest.raises(ValueError, match="integers"):
        nat.copy_env_indices(torch.tensor([0.0]), torch.tensor([1]), 4, 4)


def test_copy_envs_checks_arguments_before_any_cuda_call():
    lib = nat.load_library()
    assert lib.sr_copy_envs(None, None, None, None, 1, None) == -1
    assert lib.sr_last_error().decode() == "sr_copy_envs: null handle"


def test_every_vector_env_lists_its_per_env_state():
    import gym_softrobot_b200 as gsb
    from gym_softrobot_b200.envs.fork import ForkableVectorEnv
    for env_id, (entry, _) in gsb.VECTOR_REGISTRY.items():
        cls = gsb._load(entry)
        assert issubclass(cls, ForkableVectorEnv) and cls.PER_ENV, env_id


# ---- GPU: handle level ----------------------------------------------------------------------------------------------
def _shift_x(rows, rng, n_env, scale=0.1):
    """The reset rows of one env for every env, each whole env moved along x by its own random offset."""
    init = np.repeat(np.asarray(rows, dtype=np.float64).reshape(1, -1), n_env, axis=0)
    dx = rng.uniform(-scale, scale, n_env)
    for b in range(init.shape[1] // 9):
        init[:, 9 * b] += dx
    return init


def _random_dirs(rng, n_env):
    """Reset rows of rods at the origin with a random direction and a random normal perpendicular to it."""
    init = np.zeros((n_env, 9))
    for e in range(n_env):
        d = rng.normal(size=3); d /= np.linalg.norm(d)
        m = np.cross(d, rng.normal(size=3)); m /= np.linalg.norm(m)
        init[e, 3:6], init[e, 6:9] = d, m
    return init


def _plain_rod(n_env, n, dtype=nat.DTYPE_F64):
    return nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n, dt=2e-6 * 1023 / n if n > 200 else 5e-5, base_length=1.0,
                      base_radius=0.004 if n > 200 else 0.025, density=1000.0, youngs_modulus=1e6,
                      gravity=(0.0, 0.0, -9.81), damping_constant=2e-3, bc_kind=nat.BC_ONE_END_FIXED, dtype=dtype)


def _spline_arm(n_env, n):
    from gym_softrobot_b200.envs.soft_arm_tracking import _E, _L, _R, spline_scale
    dt = 2e-4 if n <= 40 else 1e-5 * 1024 / n
    return nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n, dt=dt, base_length=_L, base_radius=_R, density=1e-3,
                      youngs_modulus=_E, damping_constant=_E * 1e-7, bc_kind=nat.BC_ONE_END_FIXED,
                      damping_before_constraints=True,
                      spline=dict(directions=(0, 1), n_ctrl=4, scale=spline_scale(n), max_rate=0.004))


def _case(name, n_env, rng):
    """(handle, reset rows, per-env inputs, substeps per launch, action range) of a named case."""
    import gym_softrobot_b200 as gsb
    from gym_softrobot_b200.envs import soft_pendulum as sp, soft_pendulum_3d as sp3, arm_single as asg
    from gym_softrobot_b200.envs.arm_push import ArmPushVectorEnv
    if name in ("pendulum", "faithful"):
        n = 50 if name == "pendulum" else 40
        h = sp._make_handle(n_env, n, 1e-4, 0, nat.MATH_FAST if name == "pendulum" else nat.MATH_FAITHFUL)
        return h, sp.pendulum_init_params(rng.random(n_env)), ("action",), 200, (-22.0, 22.0)
    if name in ("rod", "rod_fp32", "rod_cluster"):
        h = _plain_rod(n_env, 2048 if name == "rod_cluster" else 100, nat.DTYPE_F32 if name == "rod_fp32" else nat.DTYPE_F64)
        return h, _random_dirs(rng, n_env), (), 60 if name == "rod_cluster" else 200, None
    if name in ("pendulum3d", "pendulum3d_cluster"):
        n = 50 if name == "pendulum3d" else 1024
        dt = 1e-4 if n == 50 else 2e-6 * 1023 / n
        skip = int(1.0 / ((25 if n == 50 else 2500) * dt))
        h = sp3._make_handle(n_env, n, dt, skip, 0)
        return h, sp3.pendulum3d_init_params(rng.uniform(-1.0, 1.0, n_env)), ("action",), skip, (-1.0, 1.0)
    if name == "plane":
        h = asg._make_handle(n_env, 50, 7e-5, 0)
        return h, _shift_x([0, 0, 0, 1, 0, 0, 0, 0, 1], rng, n_env), ("rest_kappa",), 150, None
    if name == "plane_cluster":
        import test_long_rods_contact as tc
        kw, N, a = tc._case("ffirst", 1024)
        h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, math=nat.MATH_FAST, **kw)
        return h, _shift_x(tc._init(N, a, 1)[0], rng, n_env), ("rest_kappa",), 60, None
    if name == "snake":
        env = gsb.make_vec("ContinuumSnake-v0", n_env)
        return env.handle, _shift_x(env._init[0], rng, n_env, 0.05), ("muscle",), 500, None
    if name in ("spline", "spline_cluster"):
        n = 40 if name == "spline" else 1024
        return _spline_arm(n_env, n), _shift_x([0, 0, 0, 0, 1, 0, 0, 0, 1], rng, n_env, 10.0), ("spline",), 50 if n == 40 else 40, None
    if name == "octoflat":
        env = gsb.make_vec("OctoFlat-v0", n_env)
        return env.handle, _shift_x(env._init_row, rng, n_env), ("rest_kappa",), 142, None
    if name == "tapered":
        env = ArmPushVectorEnv(n_env, mode="continuous")
        return env.handle, _shift_x(env._init[0], rng, n_env, 0.05), ("sucker", "sucker_idx", "tm_act", "ext"), 250, None
    if name in ("reach", "arm_two"):
        env = gsb.make_vec("OctoReach-v0" if name == "reach" else "OctoArmTwo-v0", n_env)
        inputs = ("mus_act",) if name == "reach" else ("mus_act", "msucker")
        return env.handle, _shift_x(env._init[0], rng, n_env, 0.05), inputs, 200, None
    raise KeyError(name)


CASES = ["pendulum", "rod", "rod_fp32", "faithful", "pendulum3d", "plane", "snake", "spline", "octoflat", "tapered",
         "reach", "arm_two", "rod_cluster", "pendulum3d_cluster", "plane_cluster", "spline_cluster"]


def _draw(h, name, rng, act_range):
    """Random per-env inputs, leading dimension n_env."""
    N, R, n = h.n_env, h.n_rod, h.n_elem
    s = np.linspace(0.0, 1.0, n)
    if name == "action":
        return rng.uniform(*act_range, (N, h.action_dim)).astype(np.float32)
    if name == "rest_kappa":
        amp = rng.uniform(-3.0, 3.0, (N, R, 1))
        rk = np.zeros((N, R, 3, n - 1))
        rk[:, :, 0] = amp * np.sin(np.pi * rng.integers(1, 4, (N, R, 1)) * s[None, None, :n - 1] + rng.uniform(0, np.pi, (N, R, 1)))
        return rk
    if name == "ext":
        return (rng.uniform(-1e-3, 1e-3, (N, R, 3, n + 1)), rng.uniform(-1e-5, 1e-5, (N, R, 3, n)))
    if name == "sucker" or name == "tm_act":
        return rng.uniform(0.0, 1.0, (N, R))
    if name == "sucker_idx":
        return rng.integers(-n, n, (N, R)).astype(np.int32)
    if name == "mus_act":
        return rng.uniform(0.0, 1.0, (N, R, 3, n))
    if name == "msucker":
        return rng.uniform(0.0, 1.0, (N, R, 3))
    if name == "muscle":
        beta = rng.uniform(-2e-4, 2e-4, (N, 1)) * np.sin(np.pi * s)[None, :] + rng.uniform(-1e-4, 1e-4, (N, 1)) * np.sin(3 * np.pi * s)[None, :]
        return (rng.uniform(3.0, 12.0, N), beta)
    if name == "spline":
        return rng.uniform(-1.0, 1.0, (N, 3, h.cfg.spline_n_ctrl))
    raise KeyError(name)


def _take(x, rows):
    return tuple(v[rows] for v in x) if isinstance(x, tuple) else x[rows]


def _set(h, name, x):
    """Write the inputs `x` of `_draw` into the handle (the action is passed to the step instead)."""
    import torch

    def put(t, a):
        t.copy_(torch.as_tensor(np.ascontiguousarray(a)).reshape(t.shape))
    if name == "rest_kappa":
        put(h.rest_kappa_tensor(), x)
    elif name == "ext":
        f, c = h.ext_load_tensors()
        put(f, x[0]); put(c, x[1])
    elif name == "sucker":
        put(h.sucker_tensor(), x)
    elif name == "sucker_idx":
        put(h.sucker_index_tensor(), x)
    elif name == "tm_act":
        put(h.tm_activation_tensor(), x)
    elif name == "mus_act":
        put(h.muscle_activation_tensor(), x)
    elif name == "msucker":
        put(h.fixed_sucker_tensor(), x)
    elif name == "muscle":
        mu = h.muscle_tensor()
        put(mu[:, 1], x[0]); put(mu[:, 2:], x[1])
    elif name == "spline":
        put(h.spline_tensors()[0][:, :, :h.cfg.spline_n_ctrl], x)


def _buffers(h, inputs):
    """Every per-env buffer the case uses, as [n_env, -1] copies."""
    N = h.n_env
    out = {"state": h.state_tensor(), "aux": h.aux_tensor()}
    if h.cfg.has_head:
        out["head"] = h.head_tensor()
    views = {"rest_kappa": lambda: {"rest_kappa": h.rest_kappa_tensor()},
             "ext": lambda: dict(zip(("ext_force", "ext_couple"), h.ext_load_tensors())),
             "sucker": lambda: {"sucker": h.sucker_tensor()}, "sucker_idx": lambda: {"sucker_idx": h.sucker_index_tensor()},
             "tm_act": lambda: {"tm_act": h.tm_activation_tensor()}, "mus_act": lambda: {"mus_act": h.muscle_activation_tensor()},
             "msucker": lambda: {"msucker": h.fixed_sucker_tensor()}, "muscle": lambda: {"muscle": h.muscle_tensor()},
             "spline": lambda: dict(zip(("spline_points", "spline_magnitudes"), h.spline_tensors()))}
    for name in inputs:
        if name in views:
            out.update(views[name]())
    return {k: v.reshape(N, -1).clone() for k, v in out.items()}


def _step(h, action, k):
    import torch
    obs = torch.empty((h.n_env, max(h.obs_dim, 6)), dtype=torch.float32, device="cuda")
    rew = torch.empty(h.n_env, dtype=torch.float64, device="cuda")
    term = torch.empty(h.n_env, dtype=torch.uint8, device="cuda")
    a = torch.as_tensor(action, device="cuda").contiguous() if h.action_dim else None
    h.step(a, k, obs, rew, term)


def _assert_rows(a, b, rows, what):
    import torch
    for k in a:
        for e, r in enumerate(rows):
            assert torch.equal(a[k][e], b[k][r]), f"{what}: {k} of env {e} != env {r}"


def _fork_run(name):
    """Seven envs, two launches of different inputs, the fork and the swap, two more launches with every
    destination fed its source's inputs.  Checks the subject against the twin; returns the subject's final rows."""
    import torch
    rng = np.random.default_rng(11)
    h, init, inputs, K, act_range = _case(name, N_ENV, rng)
    twin, _, _, _, _ = _case(name, N_ENV, np.random.default_rng(11))
    for x in (h, twin):
        x.reset_host(init)
    for _ in range(2):
        xs = {i: _draw(h, i, rng, act_range) for i in inputs + (("action",) if h.action_dim and "action" not in inputs else ())}
        for x in (h, twin):
            for i, v in xs.items():
                _set(x, i, v)
            _step(x, xs.get("action"), K)
    before = _buffers(h, inputs)
    launches = h.launch_count
    h.copy_envs(*FORK)
    h.copy_envs(*SWAP)
    torch.cuda.synchronize()
    assert h.launch_count == launches + 4              # a gather and a scatter per copy within the handle
    after, ref = _buffers(h, inputs), _buffers(twin, inputs)
    _assert_rows(after, ref, SOURCE_OF, f"{name} right after the copy")
    _assert_rows(after, before, SOURCE_OF, f"{name} right after the copy (against the rows before it)")
    for _ in range(2):
        xs = {i: _draw(h, i, rng, act_range) for i in inputs + (("action",) if h.action_dim and "action" not in inputs else ())}
        for i, v in xs.items():
            _set(twin, i, v)
            _set(h, i, _take(v, SOURCE_OF))
        _step(twin, xs.get("action"), K)
        _step(h, _take(xs["action"], SOURCE_OF) if "action" in xs else None, K)
    torch.cuda.synchronize()
    final, ref = _buffers(h, inputs), _buffers(twin, inputs)
    _assert_rows(final, ref, SOURCE_OF, f"{name} after stepping on")
    moved = [not torch.equal(final["state"][e], after["state"][e]) for e in range(N_ENV)]
    assert all(moved), f"{name}: an env did not move after the copy"
    out = {k: v.cpu() for k, v in final.items()}
    h.close(); twin.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_forked_envs_continue_bit_for_bit(name):
    first = _fork_run(name)
    second = _fork_run(name)
    import torch
    for k in first:
        assert torch.equal(first[k], second[k]), f"{name}: {k} differs between two identical runs"


# ---- GPU: between handles -------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_one_env_onto_every_env_of_another_handle():
    import torch
    from gym_softrobot_b200.envs.soft_pendulum import _make_handle, pendulum_init_params
    rng = np.random.default_rng(3)
    plant, planner = _make_handle(1, 50, 1e-4, 0, 0), _make_handle(64, 50, 1e-4, 0, 0)
    plant.reset_host(pendulum_init_params(rng.random(1)))
    planner.reset_host(pendulum_init_params(rng.random(64)))
    for _ in range(2):
        _step(plant, rng.uniform(-22, 22, (1, 1)).astype(np.float32), 300)
        _step(planner, rng.uniform(-22, 22, (64, 1)).astype(np.float32), 300)
    launches = planner.launch_count
    planner.copy_envs(range(64), [0] * 64, src=plant)
    assert planner.launch_count == launches + 1       # one launch between two handles
    a = rng.uniform(-22, 22, (1, 1)).astype(np.float32)
    _step(plant, a, 300)
    _step(planner, np.repeat(a, 64, axis=0), 300)
    torch.cuda.synchronize()
    p, q = _buffers(plant, ()), _buffers(planner, ())
    for k in p:
        assert torch.equal(q[k], p[k].expand_as(q[k])), k
    plant.close(); planner.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(n_elem=21), dict(dtype=nat.DTYPE_F32), dict(model=nat.MODEL_SOFT_PENDULUM),
                                dict(n_rod=2)], ids=["n_elem", "dtype", "model", "n_rod"])
def test_copy_between_handles_of_other_shapes_is_rejected(kw):
    base = dict(model=nat.MODEL_ROD, n_env=4, n_elem=20, dt=1e-4, base_length=1.0, base_radius=0.05, density=1000.0,
                youngs_modulus=1e6, bc_kind=nat.BC_FREE)
    a, b = nat.Handle(**base), nat.Handle(**{**base, **kw})
    for dst, src in ((a, b), (b, a)):
        with pytest.raises(nat.SoftRodError, match="sr_copy_envs: the two handles were created with different shapes"):
            dst.copy_envs([0], [0], src=src)
    a.close(); b.close()


@pytest.mark.gpu
def test_copy_between_devices_is_rejected():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from gym_softrobot_b200.envs.soft_pendulum import _make_handle
    a, b = _make_handle(2, 50, 1e-4, 0, 0), _make_handle(2, 50, 1e-4, 1, 0)
    with pytest.raises(nat.SoftRodError, match="different devices"):
        a.copy_envs([0], [1], src=b)
    a.close(); b.close()


@pytest.mark.gpu
def test_rest_curvature_the_source_never_allocated_is_zero():
    """sr_get_rest_kappa allocates on first use, zeroed: a source without the buffer copies zeros into the destination
    rows, and a destination without it gets one holding the source's rows."""
    import torch
    from gym_softrobot_b200.envs.arm_single import _make_handle
    init = np.tile([0, 0, 0, 1.0, 0, 0, 0, 0, 1.0], (3, 1))
    bare, shaped = _make_handle(3, 50, 7e-5, 0), _make_handle(3, 50, 7e-5, 0)
    for h in (bare, shaped):
        h.reset_host(init)
    shaped.rest_kappa_tensor()[:] = 2.0
    shaped.copy_envs([1], [0], src=bare)
    rk = shaped.rest_kappa_tensor()
    assert float(rk[1].abs().max()) == 0.0 and float(rk[0].min()) == 2.0 and float(rk[2].min()) == 2.0
    fresh = _make_handle(3, 50, 7e-5, 0)
    fresh.reset_host(init)
    fresh.copy_envs([2], [0], src=shaped)
    rk = fresh.rest_kappa_tensor()
    assert float(rk[2].min()) == 2.0 and float(rk[:2].abs().max()) == 0.0
    torch.cuda.synchronize()
    for h in (bare, shaped, fresh):
        h.close()


# ---- GPU: vector envs -----------------------------------------------------------------------------------------------
IDS = ["SoftPendulum-v0", "SoftPendulum3D-v0", "OctoArmSingle-v0", "OctoFlat-v0", "OctoFlatLite-v0",
       "ContinuumSnake-v0", "SoftArmTracking-v0", "OctoCrawl-v0", "OctoArmPush-v0", "OctoArmPush-v1",
       "OctoArmPullWeight-v0", "OctoReach-v0", "OctoArmTwo-v0"]
FAST_KW = {"OctoArmSingle-v0": dict(recording_fps=100), "OctoFlat-v0": dict(recording_fps=100),
           "OctoFlatLite-v0": dict(recording_fps=100)}
# a final time inside the cross-env window: truncation on env-step 6 (SoftArmTracking-v0: 500, fixed)
SHORT_KW = {"SoftPendulum-v0": dict(final_time=0.2), "SoftPendulum3D-v0": dict(final_time=0.2),
            "OctoArmSingle-v0": dict(final_time=0.05), "OctoFlat-v0": dict(final_time=0.05),
            "OctoFlatLite-v0": dict(final_time=0.05), "SoftArmTracking-v0": {}, "OctoCrawl-v0": dict(final_time=0.2),
            "OctoArmPush-v0": dict(final_time=0.125), "OctoArmPush-v1": dict(final_time=0.125),
            "OctoArmPullWeight-v0": dict(final_time=0.125), "OctoReach-v0": dict(final_time=0.2),
            "OctoArmTwo-v0": dict(final_time=0.2)}


def _actions(sp, n, rng, scale=1.0):
    """n random actions of the space; `scale` < 1 keeps them to that share of the range around its middle."""
    import torch
    if hasattr(sp, "n"):
        return torch.as_tensor(rng.integers(0, sp.n, n), device="cuda")
    u = 0.5 + scale * (rng.uniform(0.0, 1.0, size=(n,) + sp.shape) - 0.5)
    return torch.as_tensor((sp.low + (sp.high - sp.low) * u).astype(sp.dtype), device="cuda")


def _rows(x, rows):
    return {k: v[rows] for k, v in x.items()} if isinstance(x, dict) else x[rows]


def _eq_rows(x, a, b, what):
    import torch
    if isinstance(x, dict):
        for k in x:
            _eq_rows(x[k], a, b, f"{what}[{k}]")
        return
    assert torch.equal(x[a], x[b]), what


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", IDS)
def test_vector_env_forks_within_the_batch(env_id):
    import gym_softrobot_b200 as gsb
    env = gsb.make_vec(env_id, 6, autoreset=False, **FAST_KW.get(env_id, {}))
    env.reset(seed=5)
    rng = np.random.default_rng(1)
    for _ in range(2):
        env.step(_actions(env.single_action_space, 6, rng))
    dst, src = [3, 4, 5], [0, 1, 0]
    env.copy_envs(dst, src)
    for _ in range(3):
        act = _actions(env.single_action_space, 6, rng)
        act[dst] = act[src]
        obs, rew, term, trunc, info = env.step(act)
        for d, s in zip(dst, src):
            for what, x in (("obs", obs), ("reward", rew), ("terminated", term), ("truncated", trunc)):
                _eq_rows(x, d, s, f"{env_id} {what} env {d} vs {s}")
            if "time" in info:
                _eq_rows(info["time"], d, s, f"{env_id} time env {d} vs {s}")
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", [i for i in IDS if i != "ContinuumSnake-v0"])
def test_vector_env_forks_from_another_vector_env(env_id):
    """A one-env plant stepped k1 times is copied onto every env of a four-env planner stepped k2 != k1 times: each
    copy then truncates on the plant's step (the step counts travel with the fork) and matches it bit for bit."""
    import torch
    import gym_softrobot_b200 as gsb
    kw = {**FAST_KW.get(env_id, {}), **SHORT_KW[env_id]}
    plant, planner = gsb.make_vec(env_id, 1, autoreset=False, **kw), gsb.make_vec(env_id, 4, autoreset=False, **kw)
    plant.reset(seed=2); planner.reset(seed=9)
    rng = np.random.default_rng(4)
    # (SoftArmTracking-v0 truncates on env-step 500; full-range noise for that long can blow its arm up)
    k1, scale = (497, 0.3) if env_id == "SoftArmTracking-v0" else (3, 1.0)
    for _ in range(k1):
        plant.step(_actions(plant.single_action_space, 1, rng, scale))
    planner.step(_actions(planner.single_action_space, 4, rng, scale))
    planner.copy_envs(range(4), [0] * 4, src=plant)
    truncated_at = None
    for w in range(5):
        a = _actions(plant.single_action_space, 1, rng, scale)
        o1, r1, t1, x1, i1 = plant.step(a)
        o4, r4, t4, x4, i4 = planner.step(a.repeat_interleave(4, dim=0) if a.dim() == 1 else a.repeat(4, 1))
        for e in range(4):
            for what, p, q in (("obs", o1, o4), ("reward", r1, r4), ("terminated", t1, t4), ("truncated", x1, x4)):
                if isinstance(p, dict):
                    assert all(torch.equal(p[k][0], q[k][e]) for k in p), f"{env_id} {what} env {e} step {w}"
                else:
                    assert torch.equal(p[0], q[e]), f"{env_id} {what} env {e} step {w}"
        if truncated_at is None and bool(x1[0]):
            truncated_at = w
    assert truncated_at is not None, f"{env_id}: the plant did not truncate inside the window"
    plant.close(); planner.close()


@pytest.mark.gpu
def test_snake_copies_only_between_vector_envs_at_the_same_clock():
    import torch
    import gym_softrobot_b200 as gsb
    a, b = gsb.make_vec("ContinuumSnake-v0", 2, autoreset=False), gsb.make_vec("ContinuumSnake-v0", 2, autoreset=False)
    a.reset(); b.reset()
    act = torch.tensor([[3.4e-3, 3.3e-3, 4.2e-3, 2.6e-3, 3.6e-3, 3.5e-3, 0.97]], device="cuda").repeat(2, 1)
    a.step(act)
    with pytest.raises(ValueError, match="same clock"):
        b.copy_envs([0], [1], src=a)
    b.step(act)
    b.copy_envs([0], [1], src=a)                           # the same instant: allowed
    o1, *_ = a.step(act)
    o2, *_ = b.step(act)
    assert torch.equal(o1[1], o2[0])
    a.close(); b.close()


@pytest.mark.gpu
def test_vector_env_rejects_a_source_of_another_class():
    import gym_softrobot_b200 as gsb
    a, b = gsb.make_vec("SoftPendulum-v0", 2, autoreset=False), gsb.make_vec("SoftPendulum3D-v0", 2, autoreset=False)
    with pytest.raises(ValueError, match="not a SoftPendulumVectorEnv"):
        a.copy_envs([0], [0], src=b)
    a.close(); b.close()


@pytest.mark.gpu
def test_vector_env_asks_for_a_reset_before_a_copy():
    """OctoArmSingle-v0 keeps its previous curvature, centre of mass and distance from its first reset on."""
    import gym_softrobot_b200 as gsb
    a = gsb.make_vec("OctoArmSingle-v0", 2, autoreset=False, recording_fps=100)
    with pytest.raises(ValueError, match="reset"):
        a.copy_envs([0], [1])
    a.reset()
    a.copy_envs([0], [1])
    a.close()
