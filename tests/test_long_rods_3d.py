"""SoftPendulum3D-v0 rods of 512-4095 elements on thread-block clusters (the filter model in the cluster layout of
rod_kernel_lean.cuh, DESIGN.md §4.1): the order-7 Laplace filter and the moving base across CTAs.

The filter model's substep in the cluster layout must give the bits of its CTA layout (the one-CTA filter kernel) where
both exist (512-767 elements, where SOFTROD_LEAN_CLUSTER=1 forces it), and match the C oracle from 768 elements on,
where it is the only lean filter kernel (the CTA layout would need a 1024-thread CTA, whose shared memory it overflows).

CPU: sr_create admits SoftPendulum3D-v0's model at 1024-4095 elements, and nothing else of that model; the C oracle
steps such a rod.
GPU: each kernel setting runs in a subprocess of its own (the settings are read once per process), and the saved
outputs are compared: the forced cluster kernel against the CTA layout, the default (cluster) pair against the safe kernel
alone (SOFTROD_FASTPATH=0) and the C oracle."""
import ctypes as C
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from test_long_rods import LONG_ONLY, ORACLE_FIELDS, _fields

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

EQ_SIZES = (512, 513, 517, 600, 700, 767)   # 512: the tip alone in rank 1; 517: right ghosts across the boundary
EQ_BATCHES = (("small", 7), ("big", 300))
# C = 2 ... 8; 768-1023: the cluster layout is the default; 1024: the last rank holds only the tip node
LONG_SIZES = (768, 1000, 1023, 1024, 1026, 1535, 2047, 2048, 4095)
STEP_FPS = 2500                     # step_skip = int(1 / (2500 * time_step)) substeps per env-step (400 at n = 2048)
STEPS = 2                           # env-steps (launches) per case
CLIP = 0.4995                       # start of the envs whose base is driven into the +-0.5 clip
# test_long_rods' kink (its _kink): n = 2047, envs 1 and 3 of 5 turned by 45 degrees from element 1200 (inside rank 2) /
# 512 (across the boundary between ranks 0 and 1); launches of 3 substeps, before the kink springs back into range
KINK_ENVS, KINK_LAUNCHES = 5, (3, 3, 3, 3)


def _dt(n):
    """time_step for an n-element rod: the stable step shrinks with the element length."""
    return 2e-6 * 1023 / n


def _step_skip(n):
    """Substeps per env-step, as the envs and the oracle compute them from recording_fps."""
    return int(1.0 / (STEP_FPS * _dt(n)))


def _tilts(n, n_env):
    return np.random.default_rng(n + n_env).uniform(-1.0, 1.0, n_env)


def _actions(rng, n_env, steps):
    """Random +-1 on both axes; every third env pushes +x / -y all the way (into the clip, see _clip_envs)."""
    a = rng.choice(np.float32([-1.0, 1.0]), (steps, n_env, 2))
    a[:, ::3] = np.float32([1.0, -1.0])
    return a


# ---- CPU -----------------------------------------------------------------------------------------------------------
def _cfg(**kw):
    from gym_softrobot_b200 import _native as nat
    cfg = nat.SrConfig()
    cfg.struct_size = C.sizeof(nat.SrConfig)
    cfg.model, cfg.n_env, cfg.n_elem, cfg.bc_kind = nat.MODEL_SOFT_PENDULUM_3D, 4, 2048, nat.BC_MOVING_BASE
    cfg.laplace_filter_order = 7
    cfg.dt, cfg.base_length, cfg.base_radius, cfg.density, cfg.youngs_modulus = _dt(2048), 1.0, 0.1, 4000.0, 1e6
    cfg.gravity[:] = [0.0, 0.0, -9.80665]
    cfg.damping_constant = 1.0
    cfg.base_step, cfg.base_limit, cfg.base_move_period = 1e-3, 0.5, 400 * _dt(2048)
    for k, v in kw.items():
        setattr(cfg, k, v)
    return cfg


@pytest.mark.parametrize("kw,msg", [
    (dict(laplace_filter_order=0), LONG_ONLY),
    (dict(laplace_filter_order=5), LONG_ONLY),
    (dict(point_force_on_base=1), LONG_ONLY),
    (dict(dtype=1), LONG_ONLY),                                   # FP32 storage
    (dict(contact_on=1, slip_velocity_tol=1e-4), LONG_ONLY),
    (dict(n_elem=4096), "n_elem <= 4095"),
], ids=["filter0", "filter5", "point_force", "fp32", "contact", "4096"])
def test_create_rejects_3d_long_rods_it_does_not_build(kw, msg):
    """Checked with the other arguments, ahead of the device check; the message names what is built, the 3D model
    included."""
    from gym_softrobot_b200 import _native as nat
    lib = nat.load_library()
    h = C.c_void_p()
    rc = lib.sr_create(C.byref(_cfg(**kw)), C.byref(h))
    assert rc == -1 and not h.value
    err = lib.sr_last_error().decode()
    assert msg in err
    if msg == LONG_ONLY:
        assert "SR_MODEL_SOFT_PENDULUM_3D with SR_BC_MOVING_BASE and laplace_filter_order = 7" in err


@pytest.mark.parametrize("n", (2048, 4095))
def test_create_accepts_3d_long_rods(n):
    """SoftPendulum3D-v0's model at n = 2048 and 4095 passes every argument check: no GPU, the device error; a B200,
    a handle."""
    from gym_softrobot_b200 import _native as nat
    lib = nat.load_library()
    h = C.c_void_p()
    rc = lib.sr_create(C.byref(_cfg(n_elem=n, dt=_dt(n), base_move_period=400 * _dt(n))), C.byref(h))
    assert rc in (0, -3), lib.sr_last_error().decode()
    if rc == 0:
        lib.sr_destroy(h)


def test_oracle_steps_3d_long_rod():
    """OracleSoftPendulum3D at n_elems = 2048 (time_step 1e-6, 400 substeps per env-step) over 10 env-steps of random
    +-1 actions: finite state, no termination."""
    import rod_oracle as ro
    e = ro.OracleSoftPendulum3D(n_elems=2048, time_step=_dt(2048), recording_fps=STEP_FPS)
    assert e.step_skip == 400
    e.reset(seed=3)
    for a in np.random.default_rng(3).choice(np.float32([-1.0, 1.0]), (10, 2)):
        obs, rew, term, trunc, info = e.step(a)
        assert np.isfinite(obs).all() and np.isfinite(rew) and not term and not trunc
    assert np.isfinite(e.rod.position_collection).all() and np.isfinite(e.rod.omega_collection).all()
    e.rod.close()


# ---- the GPU worker --------------------------------------------------------------------------------------------------
_WORKER = r"""
import os, sys
import numpy as np
root, cases, out = sys.argv[1], sys.argv[2].split(","), sys.argv[3]
sys.path[:0] = [root, os.path.join(root, "tests")]
import torch
import test_long_rods_3d as t3
import test_long_rods as tl
from gym_softrobot_b200 import _native as nat
from gym_softrobot_b200.envs.soft_pendulum_3d import _make_handle, pendulum3d_init_params
res = {}

def make(n, n_env, clip=False):
    h = _make_handle(n_env, n, t3._dt(n), t3._step_skip(n), 0)
    init = pendulum3d_init_params(t3._tilts(n, n_env))
    if clip:
        init[::3, 0], init[::3, 1] = t3.CLIP, -t3.CLIP
    h.reset_host(init)
    if clip:      # the base controller starts where the rod's base is
        aux = h.aux_tensor()
        aux[::3, 0], aux[::3, 1] = t3.CLIP, -t3.CLIP
        torch.cuda.synchronize()
    return h

def counts(h):
    return np.array([h.fallback_count(), *h.fallback_causes(), h.launch_count])

def run(key, h, actions, substeps=None):
    for li, a in enumerate(actions):
        o, r, t = h.step_host(a, substeps[li] if substeps else t3._step_skip(h.n_elem))
        res[f"{key}/obs{li}"], res[f"{key}/rew{li}"], res[f"{key}/term{li}"] = o.copy(), r.copy(), t.copy()
        res[f"{key}/state{li}"] = h.state_tensor().cpu().numpy()
        res[f"{key}/aux{li}"] = h.aux_tensor().cpu().numpy()
        res[f"{key}/counts{li}"] = counts(h)
    res[f"{key}/counts"] = counts(h)

if "eq" in cases:
    for n in t3.EQ_SIZES:
        for size, n_env in t3.EQ_BATCHES:
            h = make(n, n_env, clip=True)
            run(f"eq{n}/{size}", h, t3._actions(np.random.default_rng(n + n_env), n_env, t3.STEPS))
            h.close()

if "long" in cases:
    for n in t3.LONG_SIZES:
        h = make(n, 3)
        run(f"long{n}", h, t3._actions(np.random.default_rng(n), 3, t3.STEPS))
        h.close()
    h = make(2048, 3)
    res["layout"] = np.array([getattr(h.state_view(), f) for f in ("f_position", "f_velocity", "f_director", "f_omega",
                                                                   "f_tangents", "f_kappa", "f_sigma", "f_dilatation")])
    errs = []
    for call in (h.rest_kappa_tensor, h.ext_load_tensors):
        try:
            call()
            errs.append("")
        except nat.SoftRodError as ex:
            errs.append(str(ex))
    res["getter_errors"] = np.array(errs)
    # sr_observe at this length equals the observation of the step that produced the state
    a = np.float32([[1.0, -1.0]] * 3)
    o, _, _ = h.step_host(a, 400)
    obs = torch.empty((3, 9), dtype=torch.float32, device="cuda")
    h.observe(torch.as_tensor(a, device="cuda").contiguous(), obs)
    res["observe"], res["observe_step"] = obs.cpu().numpy(), o.copy()
    h.close()

if "kink" in cases:
    h = make(tl.KINK_N, t3.KINK_ENVS)
    fl = h.fields()
    x, Q = (fl[k].cpu().numpy() for k in ("position_collection", "director_collection"))
    tl._kink(x, Q)
    for k, arr in (("position_collection", x), ("director_collection", Q)):
        fl[k][:] = torch.as_tensor(arr, device="cuda")
    torch.cuda.synchronize()
    L = len(t3.KINK_LAUNCHES)
    run("kink", h, np.zeros((L, t3.KINK_ENVS, 2), np.float32), t3.KINK_LAUNCHES)
    h.close()

if "nan" in cases:
    for key in ("nan", "nonan"):     # the same handle and actions with and without a NaN in env 2
        h = make(2048, 4)
        if key == "nan":
            v = h.fields()["velocity_collection"].cpu().numpy()
            v[2, 1, h.n_elem] = np.nan          # the tip node: the last thread of the last rank
            h.fields()["velocity_collection"][:] = torch.as_tensor(v, device="cuda")
            torch.cuda.synchronize()
        run(key, h, t3._actions(np.random.default_rng(4), 4, 1))
        h.close()

np.savez(out, **res)
"""

# SOFTROD_* settings of a worker process -> the cases it runs
SETTINGS = {"default": ({}, "eq,long,kink,nan"), "cluster": ({"SOFTROD_LEAN_CLUSTER": "1"}, "eq"),
            "safe": ({"SOFTROD_FASTPATH": "0"}, "kink")}
_KNOBS = ("SOFTROD_LEAN_CLUSTER", "SOFTROD_FASTPATH")


@pytest.fixture(scope="module")
def worker(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("long_rods_3d")
    script = tmp / "long_rods_3d_worker.py"
    script.write_text(_WORKER)

    @functools.lru_cache(maxsize=None)
    def get(setting):
        extra, cases = SETTINGS[setting]
        env = {k: v for k, v in os.environ.items() if k not in _KNOBS}
        env.update(extra)
        out = tmp / f"{setting}.npz"
        res = subprocess.run([sys.executable, str(script), ROOT, cases, str(out)], stdout=subprocess.PIPE,
                             stderr=subprocess.STDOUT, text=True, env=env, timeout=3000)
        assert res.returncode == 0, res.stdout[-3000:]
        return dict(np.load(out))
    return get


# ---- 1 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", EQ_SIZES)
def test_cluster_filter_kernel_gives_the_bits_of_variant_4(worker, n):
    """SOFTROD_LEAN_CLUSTER=1 (the filter model on clusters, two CTAs per rod) against the default one-CTA filter kernel
    (the CTA layout, 544 / 768-thread CTAs), 7 and 300 envs, random +-1 actions with every third env's base starting next
    to the (0.5, -0.5) corner and driven into the clip: after each of two env-steps the whole state block (all 32 fields), aux
    (base controller and tilt), the observations, rewards and terminated flags are equal bit for bit, with no range
    fallback in either."""
    ref, cl = worker("default"), worker("cluster")
    for size, _ in EQ_BATCHES:
        key = f"eq{n}/{size}"
        for li in range(STEPS):
            for f in ("state", "aux", "obs", "rew", "term"):
                a, b = ref[f"{key}/{f}{li}"], cl[f"{key}/{f}{li}"]
                assert a.shape == b.shape, (key, f)
                assert np.array_equal(a, b), (key, f, li, np.argwhere(a != b)[:5])
        assert ref[f"{key}/counts"][0] == 0 and cl[f"{key}/counts"][0] == 0, (key, ref[f"{key}/counts"], cl[f"{key}/counts"])
        assert not cl[f"{key}/term{STEPS - 1}"].any()
        aux = cl[f"{key}/aux{STEPS - 1}"]
        assert (aux[::3, 0] == 0.5).all() and (aux[::3, 1] == -0.5).all(), aux[::3, :2]    # the clip was reached


# ---- 2 -------------------------------------------------------------------------------------------------------------
def _oracle_env(n, tilt):
    import rod_oracle as ro
    e = ro.OracleSoftPendulum3D(n_elems=n, time_step=_dt(n), recording_fps=STEP_FPS)
    e.reset(tilt_deg=tilt)
    return e


class _Rod:
    """An OracleSoftPendulum3D after reset, seen as its rod (for one_ulp_divergence)."""

    def __init__(self, n, tilt):
        self.env = _oracle_env(n, tilt)

    def __getattr__(self, k):
        return getattr(self.env.rod, k)

    def close(self):
        self.env.rod.close()


def _check_vs_oracle(res, key, n, tilts, actions, envs, what):
    """Every field, the observation (2 float32 ulp), reward and tilt (1e-9) after each env-step against the C oracle."""
    from test_parity_gpu import assert_state_close, one_ulp_divergence, rate_floors
    layout = res["layout"]
    for e in envs:
        o = _oracle_env(n, tilts[e])
        refs = []
        for a in actions[:, e]:
            oo, orew, ote, _, info = o.step(a)
            refs.append(({k: getattr(o.rod, k).copy() for k in ORACLE_FIELDS}, oo, orew, ote, info["tilt"]))
        o.rod.close()

        def advance(rod):
            for a in actions[:, e]:
                rod.env.step(a)
        sens = one_ulp_divergence(lambda: _Rod(n, tilts[e]), advance, refs[-1][0])
        for li, (ref, oo, orew, ote, tilt) in enumerate(refs):
            f = _fields(res[f"{key}/state{li}"][e], layout, n)
            floors = rate_floors(1e6, 4000.0, 1.0, n, 0.1, np.abs(ref["position_collection"]).max())
            w = f"{what} env {e} after step {li}"
            for name in ORACLE_FIELDS:
                assert_state_close(f[name], ref[name], name, floors, w, measured=sens)
            np.testing.assert_array_max_ulp(res[f"{key}/obs{li}"][e], oo, maxulp=2)
            rew = float(res[f"{key}/rew{li}"][e])
            assert abs(rew - orew) <= 1e-9 * max(1.0, abs(orew)), (w, rew, orew)
            assert abs(float(res[f"{key}/aux{li}"][e, 6]) - tilt) <= 1e-9, (w, res[f"{key}/aux{li}"][e, 6], tilt)
            assert bool(res[f"{key}/term{li}"][e]) == ote, w


@pytest.mark.gpu
@pytest.mark.parametrize("n", LONG_SIZES)
def test_3d_long_rods_vs_c_oracle(worker, n):
    """SoftPendulum3D-v0 rods of 768-4095 elements (clusters of 2 ... 8 CTAs), three envs, two env-steps of random +-1
    actions, against OracleSoftPendulum3D: all eight fields within the 1e-9 rule of test_parity_gpu or 20x the
    oracle's own one-ulp divergence, the observation within 2 float32 ulp, reward and tilt within 1e-9; no fallback,
    and the launches of the cluster pair."""
    res = worker("default")
    key = f"long{n}"
    _check_vs_oracle(res, key, n, _tilts(n, 3), _actions(np.random.default_rng(n), 3, STEPS), range(3), f"n={n}")
    cnt = res[f"{key}/counts"]
    assert cnt[0] == 0 and cnt[4] == 1 + 2 * STEPS, cnt      # reset + (fast-only, fallback) per step


@pytest.mark.gpu
def test_3d_long_rod_getters(worker):
    """Rest curvature and external loads are refused at these lengths; sr_observe reads the rod across all ranks and
    gives the observation of the step that produced the state."""
    res = worker("default")
    assert "rest curvature is built for n_elem <= 1023" in res["getter_errors"][0]
    assert "external loads are built for" in res["getter_errors"][1]
    assert np.array_equal(res["observe"], res["observe_step"])


# ---- 3 -------------------------------------------------------------------------------------------------------------
API_N, API_STEPS = 2048, 10


def _api_kw():
    return dict(n_elems=API_N, time_step=_dt(API_N), recording_fps=STEP_FPS)


def _assert_step_close(state, obs, rew, term, trunc, tilt, o, oo, orew, ote, otr, otilt, what, sens):
    from test_parity_gpu import assert_state_close, rate_floors
    floors = rate_floors(1e6, 4000.0, 1.0, API_N, 0.1, np.abs(o.rod.position_collection).max())
    for name in ORACLE_FIELDS:
        assert_state_close(state[name], getattr(o.rod, name), name, floors, what, measured=sens)
    np.testing.assert_array_max_ulp(np.asarray(obs, np.float32), oo, maxulp=2)
    assert abs(float(rew) - orew) <= 1e-9 * max(1.0, abs(orew)), (what, float(rew), orew)
    assert abs(float(tilt) - otilt) <= 1e-9, (what, float(tilt), otilt)
    assert (bool(term), bool(trunc)) == (ote, otr), what


class _SeedRod:
    def __init__(self, seed):
        import rod_oracle as ro
        self.env = ro.OracleSoftPendulum3D(**_api_kw())
        self.env.reset(seed=seed)

    def __getattr__(self, k):
        return getattr(self.env.rod, k)

    def close(self):
        self.env.rod.close()


def _sensitivity(seed, actions):
    from test_parity_gpu import one_ulp_divergence
    o = _SeedRod(seed)
    for a in actions:
        o.env.step(a)
    ref = {k: getattr(o, k).copy() for k in ORACLE_FIELDS}
    o.close()

    def advance(rod):
        for a in actions:
            rod.env.step(a)
    return one_ulp_divergence(lambda: _SeedRod(seed), advance, ref)


@pytest.mark.gpu
def test_soft_pendulum_3d_2048_single_env_vs_oracle():
    """gsb.make("SoftPendulum3D-v0", n_elems=2048) resets and steps 10 env-steps of random +-1 actions as
    OracleSoftPendulum3D does."""
    import gym_softrobot_b200 as gsb
    import rod_oracle as ro
    env = gsb.make("SoftPendulum3D-v0", **_api_kw())
    o = ro.OracleSoftPendulum3D(**_api_kw())
    obs, _ = env.reset(seed=5)
    o_obs, _ = o.reset(seed=5)
    np.testing.assert_array_max_ulp(obs, o_obs, maxulp=2)
    actions = np.random.default_rng(5).choice(np.float32([-1.0, 1.0]), (API_STEPS, 2))
    sens = _sensitivity(5, actions)
    for i, a in enumerate(actions):
        obs, rew, te, tr, info = env.step(a)
        oo, orew, ote, otr, oinfo = o.step(a)
        _assert_step_close(env.rod_state(), obs, rew, te, tr, info["tilt"], o, oo, orew, ote, otr, oinfo["tilt"],
                           f"step {i}", sens)
    env.close()
    o.rod.close()


@pytest.mark.gpu
def test_soft_pendulum_3d_2048_vector_env_vs_oracle():
    """gsb.make_vec("SoftPendulum3D-v0", 64, n_elems=2048) over 10 env-steps against the oracle (6 of the envs), with
    envs 3, 17 and 40 reset through sr_reset's env_idx after step 4: the others carry on as the oracle does, and the
    reset envs step on exactly as the envs of a fresh handle reset from the same rows (state block, aux, observations,
    rewards and flags bit for bit)."""
    import torch
    import gym_softrobot_b200 as gsb
    import rod_oracle as ro
    from gym_softrobot_b200.envs.soft_pendulum_3d import _make_handle, pendulum3d_init_params
    n_env, check, reset_ids = 64, (0, 3, 17, 40, 50, 63), (3, 17, 40)
    vec = gsb.make_vec("SoftPendulum3D-v0", n_env, autoreset=False, **_api_kw())
    obs, _ = vec.reset(seed=11)
    oracles = {e: ro.OracleSoftPendulum3D(**_api_kw()) for e in check}
    for e, o in oracles.items():
        np.testing.assert_array_max_ulp(obs[e].cpu().numpy(), o.reset(seed=11 + e)[0], maxulp=2)
    actions = np.random.default_rng(11).choice(np.float32([-1.0, 1.0]), (API_STEPS, n_env, 2))
    sens = {e: _sensitivity(11 + e, actions[:, e]) for e in check}
    init = pendulum3d_init_params(np.random.default_rng(99).uniform(-1.0, 1.0, len(reset_ids)))
    fresh = _make_handle(len(reset_ids), API_N, _dt(API_N), vec.step_skip, 0)
    fresh.reset_host(init)
    ids = list(reset_ids)
    for i in range(API_STEPS):
        if i == 5:
            idx = torch.as_tensor(reset_ids, dtype=torch.int32, device="cuda")
            vec.handle.reset(torch.as_tensor(init, device="cuda").contiguous(), idx)
        a = actions[i]
        obs, rew, te, tr, info = vec.step(torch.as_tensor(a, device="cuda"))
        f = {k: v.cpu().numpy() for k, v in vec.fields().items()}
        tilt = info["tilt"].cpu().numpy()
        for e, o in oracles.items():
            if e in reset_ids and i >= 5:
                continue
            oo, orew, ote, otr, oinfo = o.step(a[e])
            _assert_step_close({k: f[k][e] for k in ORACLE_FIELDS}, obs[e].cpu().numpy(), rew[e], te[e], tr[e], tilt[e],
                               o, oo, orew, ote, otr, oinfo["tilt"], f"env {e} step {i}", sens[e])
        if i >= 5:
            fo, fr, ft = fresh.step_host(np.ascontiguousarray(a[ids]), vec.step_skip)
            st, fst = vec.handle.state_tensor().cpu().numpy(), fresh.state_tensor().cpu().numpy()
            assert np.array_equal(st[ids], fst), (i, np.argwhere(st[ids] != fst)[:5])
            assert np.array_equal(vec.handle.aux_tensor().cpu().numpy()[ids], fresh.aux_tensor().cpu().numpy())
            assert np.array_equal(obs[ids].cpu().numpy(), fo) and np.array_equal(rew[ids].cpu().numpy(), fr)
            assert np.array_equal(te[ids].cpu().numpy(), ft.astype(bool))
    fresh.close()
    vec.close()
    for o in oracles.values():
        o.rod.close()


# ---- 4 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_3d_range_fallback_across_ctas(worker):
    """n = 2047 (clusters of 4), still base, one env kinked by 45 degrees at element 1200 (inside rank 2), one at
    elements 511 / 512 (across the boundary between ranks 0 and 1).  The fast-only kernel flags both envs in every
    step, with cause "bend" only; the flagged envs equal the safe kernel alone (SOFTROD_FASTPATH=0) bit for bit, and
    the others are untouched by the fallback (the same bits as the safe kernel's too)."""
    res, safe = worker("default"), worker("safe")
    L = len(KINK_LAUNCHES)
    for li in range(L):
        for f in ("state", "aux", "obs", "rew", "term"):
            a, b = res[f"kink/{f}{li}"], safe[f"kink/{f}{li}"]
            assert np.array_equal(a, b), (f, li, np.argwhere(a != b)[:5])
    first = res["kink/counts0"]
    assert list(first[:4]) == [2, 0, 2, 0], first       # both envs, once, for the bend (total, rotation, bend, stretch)
    cnt = res["kink/counts"]
    assert cnt[0] == cnt[2] and cnt[1] == 0 and cnt[3] == 0 and cnt[0] <= 2 * L, cnt
    assert cnt[4] == 1 + 2 * L and safe["kink/counts"][4] == 1 + L, (cnt, safe["kink/counts"])
    assert np.isfinite(res[f"kink/state{L - 1}"]).all()


# ---- 5 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_3d_nan_in_the_last_rank_terminates_that_env_only(worker):
    """A NaN in the tip's velocity (the last thread of the last CTA) reaches rank 0's lead: env 2 is terminated with
    reward -50 and no other env; the other envs' state, aux (base controller and tilt), observations and rewards are
    those of the same run without the NaN, bit for bit."""
    res = worker("default")
    assert list(res["nan/term0"]) == [0, 0, 1, 0], res["nan/term0"]
    assert res["nan/rew0"][2] == -50.0 and not res["nonan/term0"].any()
    ok = [0, 1, 3]
    for f in ("state", "aux", "obs", "rew"):
        assert np.array_equal(res[f"nan/{f}0"][ok], res[f"nonan/{f}0"][ok]), f
