"""SoftArmTracking-v0's spline-torque rods of 512-4095 elements on thread-block clusters (the spline model in the cluster
layout of rod_kernel_lean.cuh, DESIGN.md §4.1): MuscleTorquesWithVaryingBetaSplines, its rate-limited control values
and its arc-length prefix sum across the CTAs of a cluster.

One rod spans C = ceil((n + 1) / 512) CTAs of a cluster.  The cluster kernel must give the bits of the one-CTA spline
kernel where both exist (SOFTROD_LEAN_CLUSTER=1 forces it for 512-1023 elements), and match the C oracle above 1023
elements, where it is the only kernel.

CPU: sr_create admits 1024-4095 elements for the spline model and rejects it combined with anything the cluster layout
does not build; the C oracle steps the refined SoftArmTracking arm; the env's step count and truncation follow its
time step.
GPU: each kernel setting runs in a subprocess of its own (the settings are read once per process), and the saved
outputs are compared, as in test_long_rods.py."""
import ctypes as C
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from test_long_rods import LONG_ONLY, ORACLE_FIELDS, _fields
from test_long_rods_contact import LONG_3D

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BC_FREE, BC_ONE_END_FIXED, BC_PENDULUM_SLIDER = 0, 1, 2     # (= _native / rod_oracle)
INF = float("inf")

EQ_SIZES = (512, 513, 600, 767, 1000, 1023)   # 512: the tip node alone in rank 1; 1023: both CTAs full
EQ_BATCHES = (("small", 7), ("big", 300))      # 300 envs: more clusters than are resident at once
# name -> (end, material directions, control values, max_rate).  A rate of 0.004 per substep takes up to 500 substeps
# to reach targets in [-1, 1]: the re-fit runs in every substep of both launches.
CASES = {"free01": (BC_FREE, (0, 1), 4, INF), "clamped012rate": (BC_ONE_END_FIXED, (0, 1, 2), 5, 0.004),
         "clamped01rate": (BC_ONE_END_FIXED, (0, 1), 4, 0.004), "kink": (BC_ONE_END_FIXED, (0, 1), 4, 0.004)}
EQ_CASES = ("free01", "clamped012rate", "clamped01rate")
LAUNCHES = (150, 250)
LONG_SIZES = (1024, 1535, 2047, 2048, 3000, 4095)   # C = 3 ... 8, last CTA holding 1 ... 512 threads
LONG_CASES = ("free01", "clamped012rate")
LONG_LAUNCHES = (100, 200)
LONG_ENVS = 2
REACH_N = 2047                                 # C = 4: the last rank holds elements 1536-2046
KINK_N, KINK_ENVS, KINK_AT = 2047, 5, {1: 1200, 3: 512}   # inside rank 2 / rank 1's first element (Voronoi 511)
KINK_DEG = 60.0
# the spline model's bend map (rod_kernel_lean.cuh): the polynomial for w2 = |axial(Q_{j+1} Q_j^T - its transpose)|^2
# = 4 sin^2(theta) <= kNarrowBendW2 (rod_math.cuh, 23.07 degrees), the reference map above
NARROW_BEND_W2 = 0.6144
# one substep per launch, so that the bend is checked at every substep boundary.  (The env's arm, R = 50 mm on 0.5 mm
# elements, straightens a 60-degree kink to below the map's limit within three substeps; the thin rod of
# test_long_rods, r = 4 mm, keeps it above twice the limit for eight.)
KINK_LAUNCHES = (1,) * 8
E2E_ENVS, E2E_N, E2E_DT, E2E_STEPS, E2E_RESET = 8, 2048, 5e-6, 3, (1, 4)


def _arm(name, n):
    """Handle / oracle keyword arguments of a named case: SoftArmTracking-v0's arm (L = 1000 mm, R = 50 mm) refined to
    n elements at dt = 1e-5 x 1024 / n, its spline magnitude scaled by 40 / n (soft_arm_tracking.spline_scale); the
    "kink" case: test_long_rods' rod (L = 1 m, r = 4 mm, dt = 2e-6 x 1023 / n) with a magnitude of the order of its EI."""
    from gym_softrobot_b200.envs.soft_arm_tracking import _E, _L, _R, spline_scale
    bc, dirs, P, rate = CASES[name]
    if name == "kink":
        return dict(n_elem=n, dt=2e-6 * 1023 / n, base_length=1.0, base_radius=0.004, density=1000.0, youngs_modulus=1e6,
                    damping_constant=1e-2, bc_kind=bc, damping_before_constraints=True,
                    spline=dict(directions=dirs, n_ctrl=P, scale=1e-3, max_rate=rate))
    return dict(n_elem=n, dt=1e-5 * 1024 / n, base_length=_L, base_radius=_R, density=1e-3, youngs_modulus=_E,
                damping_constant=_E * 1e-7, bc_kind=bc, damping_before_constraints=True,
                spline=dict(directions=dirs, n_ctrl=P, scale=spline_scale(n), max_rate=rate))


def _init(n_env):
    """sr_reset rows: the env's arm, from the origin along +y, its d1 along +z."""
    return np.tile([0.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0], (n_env, 1))


def _targets(rng, n_env, P):
    return rng.uniform(-1.0, 1.0, (n_env, 3, P))


# ---- CPU -----------------------------------------------------------------------------------------------------------
def _cfg(n, **kw):
    """The env's clamped arm of n elements with spline torques in directions 0 and 1; keyword arguments set SrConfig
    fields (lists for the array fields)."""
    from gym_softrobot_b200 import _native as nat
    cfg = nat.SrConfig()
    cfg.struct_size = C.sizeof(nat.SrConfig)
    cfg.model, cfg.n_env, cfg.n_elem, cfg.bc_kind = nat.MODEL_ROD, 4, n, nat.BC_ONE_END_FIXED
    cfg.dt, cfg.base_length, cfg.base_radius, cfg.density, cfg.youngs_modulus = 5e-6, 1000.0, 50.0, 1e-3, 2e6
    cfg.damping_constant = 0.2
    cfg.spline_dir_mask, cfg.spline_n_ctrl, cfg.spline_scale, cfg.spline_max_rate = 3, 4, 1e9 * 40 / n, INF
    for k, v in kw.items():
        if isinstance(v, (list, tuple)):
            getattr(cfg, k)[:] = list(v)
        else:
            setattr(cfg, k, v)
    return cfg


@pytest.mark.parametrize("n", [2048, 4095])
@pytest.mark.parametrize("bc", [BC_FREE, BC_ONE_END_FIXED], ids=["free", "clamped"])
@pytest.mark.parametrize("mask", [3, 4, 7], ids=["d01", "d2", "d012"])
@pytest.mark.parametrize("n_ctrl", [2, 14])
def test_create_accepts_long_spline_rods(n, bc, mask, n_ctrl):
    """Free and clamped spline rods pass every argument check at 2048 and 4095 elements, for any direction set and
    2 or 14 control values: no GPU, the device error; a B200, a handle."""
    from gym_softrobot_b200 import _native as nat
    lib = nat.load_library()
    h = C.c_void_p()
    rc = lib.sr_create(C.byref(_cfg(n, bc_kind=bc, spline_dir_mask=mask, spline_n_ctrl=n_ctrl)), C.byref(h))
    assert rc in (0, -3), lib.sr_last_error().decode()
    if rc == 0:
        lib.sr_destroy(h)


@pytest.mark.parametrize("kw", [
    dict(bc_kind=BC_PENDULUM_SLIDER),
    dict(point_force_on_base=1),
    dict(dtype=1),
    dict(math=1),
    dict(contact_on=1, slip_velocity_tol=1e-4, contact_k=1e2, contact_nu=1e1, plane_normal=[0.0, 0.0, 1.0]),
    dict(muscle_on=1, muscle_period=1.0, muscle_ramp_up_time=1.0),
    dict(laplace_filter_order=7),
    dict(tip_radius=25.0),
], ids=["slider", "point-force", "fp32", "faithful", "contact", "muscle", "laplace", "tapered"])
def test_create_rejects_long_spline_rods_it_does_not_build(kw):
    """Checked ahead of the device check, with the message that names what is built: the same answer with or without
    a GPU."""
    from gym_softrobot_b200 import _native as nat
    lib = nat.load_library()
    h = C.c_void_p()
    rc = lib.sr_create(C.byref(_cfg(2048, **kw)), C.byref(h))
    assert rc == -1 and not h.value
    msg = lib.sr_last_error().decode()
    assert msg.startswith("sr_create: " + LONG_ONLY) and LONG_3D in msg, msg


def test_oracle_steps_the_refined_arm():
    """The C oracle (the GPU tests' reference) steps SoftArmTracking-v0's arm at 2048 elements and 5e-6 s with the
    scaled spline magnitude and new random targets: finite, and bending."""
    import rod_oracle as ro
    from gym_softrobot_b200.envs.soft_arm_tracking import _E, _L, _R, spline_scale
    n, dt = 2048, 5e-6
    o = ro.OracleRod(n, [0, 0, 0], [0, 1.0, 0], [0, 0, 1.0], _L, _R, 1e-3, _E, dt, damping_constant=_E * 1e-7,
                     bc_kind=ro.BC_ONE_END_FIXED, damping_before_constraints=True,
                     spline=dict(directions=(0, 1), n_ctrl=4, scale=spline_scale(n), max_rate=INF))
    rng = np.random.default_rng(0)
    for _ in range(3):
        o.spline_points[:2, :4] = rng.uniform(-1, 1, (2, 4))
        o.substeps(100)
    assert np.isfinite(o.position_collection).all() and np.isfinite(o.velocity_collection).all()
    assert np.abs(o.kappa).max() > 0 and np.abs(o.spline_magnitude[:2]).max() > 0
    o.close()


def test_arm_step_count_and_truncation_follow_the_time_step():
    """At the reference's 2e-4 s the env keeps its constants (50 substeps per env-step, truncation after 500); at 5e-6
    and 1e-6 s an env-step is still 0.01 s and truncation is the first env-step with `tick * sim_dt >= 5`."""
    from gym_softrobot_b200.envs import soft_arm_tracking as sat
    assert sat.substeps_per_step(sat._DT) == sat._UPDATE == 50
    assert sat.truncation_steps(50, sat._DT) == int(np.argmax(np.arange(0, 40000, 50) * sat._DT >= 5.0)) == 500
    for dt, update in ((5e-6, 2000), (1e-6, 10000)):
        assert sat.substeps_per_step(dt) == update
        k = sat.truncation_steps(update, dt)
        assert k * update * dt >= 5.0 and not (k - 1) * update * dt >= 5.0, (dt, k)
    assert sat.spline_scale(40) == 10 * sat._R * sat._E


# ---- the GPU worker --------------------------------------------------------------------------------------------------
_WORKER = r"""
import hashlib, os, sys
import numpy as np
root, cases, out = sys.argv[1], sys.argv[2].split(","), sys.argv[3]
sys.path[:0] = [root, os.path.join(root, "tests")]
import torch
import test_long_rods_spline as ts
from gym_softrobot_b200 import _native as nat
res = {}

def init_fields(h):
    return np.concatenate([h.fields()[k].cpu().numpy().reshape(h.n_env, -1) for k in
                           ("position_collection", "velocity_collection", "director_collection", "omega_collection")], axis=1)

def layout(h):
    return np.array([getattr(h.state_view(), f) for f in ("f_position", "f_velocity", "f_director", "f_omega",
                                                           "f_tangents", "f_kappa", "f_sigma", "f_dilatation")])

def make(name, n, n_env):
    h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, math=nat.MATH_FAST, **ts._arm(name, n))
    h.reset_host(ts._init(n_env))
    torch.cuda.synchronize()
    return h

def set_targets(h, name, tg):
    pts, _ = h.spline_tensors()
    P = ts.CASES[name][2]
    for d in ts.CASES[name][1]:
        pts[:, d, :P] = torch.as_tensor(tg[:, d], device="cuda")
    torch.cuda.synchronize()

def run(key, h, name, launches, rng, full, targets=None):
    # new random targets before every launch (or the given list of [n_env, 3, P] arrays)
    for li, k in enumerate(launches):
        set_targets(h, name, targets[li] if targets is not None else ts._targets(rng, h.n_env, ts.CASES[name][2]))
        o, r, t = h.step_host(None, k)
        res[f"{key}/obs{li}"], res[f"{key}/rew{li}"], res[f"{key}/term{li}"] = o.copy(), r.copy(), t.copy()
        st = h.state_tensor().cpu().numpy()
        pts, mags = (a.cpu().numpy() for a in h.spline_tensors())
        assert np.isfinite(st).all(), key
        if full:
            res[f"{key}/state{li}"], res[f"{key}/pts{li}"], res[f"{key}/mags{li}"] = st, pts, mags
        else:
            res[f"{key}/state{li}"] = np.array([hashlib.blake2b(e.tobytes() + p.tobytes() + m.tobytes(), digest_size=16).digest()
                                               for e, p, m in zip(st, pts, mags)])
    res[f"{key}/counts"] = np.array([h.fallback_count(), h.launch_count])

def set_fields(h, **arrays):
    fl = h.fields()
    for k, a in arrays.items():
        fl[k][:] = torch.as_tensor(a, device="cuda")
    torch.cuda.synchronize()     # (the handle steps on a stream of its own)

if "eq" in cases:
    for n in ts.EQ_SIZES:
        for size, n_env in ts.EQ_BATCHES:
            for ci, name in enumerate(ts.EQ_CASES):
                h = make(name, n, n_env)
                run(f"eq{n}/{name}/{size}", h, name, ts.LAUNCHES, np.random.default_rng(100 * n + n_env + ci), size == "small")
                h.close()

if "long" in cases:
    for n in ts.LONG_SIZES:
        for ci, name in enumerate(ts.LONG_CASES):
            h = make(name, n, ts.LONG_ENVS)
            res[f"long{n}/{name}/init"] = init_fields(h)
            run(f"long{n}/{name}", h, name, ts.LONG_LAUNCHES, np.random.default_rng(1000 * n + ci), True)
            res["layout"] = layout(h)
            h.close()

if "reach" in cases:
    h = make("free01", ts.REACH_N, ts.LONG_ENVS)
    res["reach/init"] = init_fields(h)
    run("reach", h, "free01", ts.LONG_LAUNCHES, None, True, targets=ts._reach_targets())
    h.close()

if "kink" in cases:
    h = make("kink", ts.KINK_N, ts.KINK_ENVS)
    fl = h.fields()
    x, Q = (fl[k].cpu().numpy() for k in ("position_collection", "director_collection"))
    ts._kink(x, Q)
    set_fields(h, position_collection=x, director_collection=Q)
    res["kink/init"] = init_fields(h)
    run("kink", h, "kink", ts.KINK_LAUNCHES, np.random.default_rng(5), True)
    h.close()

if "nan" in cases:
    for tag in ("clean", "nan"):
        h = make("clamped012rate", 2047, 4)
        set_targets(h, "clamped012rate", ts._targets(np.random.default_rng(9), 4, 5))
        if tag == "nan":
            v = h.fields()["velocity_collection"].cpu().numpy()
            v[2, 1, h.n_elem] = np.nan          # the tip node: the last thread of the last rank
            set_fields(h, velocity_collection=v)
        o, r, t = h.step_host(None, 20)
        pts, mags = (a.cpu().numpy() for a in h.spline_tensors())
        res[f"nan/{tag}/term"], res[f"nan/{tag}/state"] = t.copy(), h.state_tensor().cpu().numpy()
        res[f"nan/{tag}/pts"], res[f"nan/{tag}/mags"], res[f"nan/{tag}/obs"] = pts, mags, o.copy()
        h.close()

if "e2e" in cases:
    import gym_softrobot_b200 as gsb
    for mode in (1, 2):
        env = gsb.make_vec("SoftArmTracking-v0", ts.E2E_ENVS, game_mode=mode, n_elems=ts.E2E_N, time_step=ts.E2E_DT)
        obs, _ = env.reset(seed=11)
        k = f"e2e{mode}"
        res[f"{k}/update"], res[f"{k}/n_updates"] = env.update, env.n_updates
        res[f"{k}/obs_reset"], res[f"{k}/init"] = obs.cpu().numpy(), init_fields(env.handle)
        res[f"{k}/targets0"] = env._targets.cpu().numpy()
        rng = np.random.default_rng(mode)
        for s in range(ts.E2E_STEPS):
            if s == 1:   # these envs reach the end of their episode in this step: truncated, then reset in the same step()
                env.tick[list(ts.E2E_RESET)] = env.n_updates - 1
            res[f"{k}/tick{s}"] = env.tick.cpu().numpy()
            a = rng.uniform(-1.0, 1.0, (ts.E2E_ENVS, 8))
            obs, rew, term, trunc, info = env.step(torch.as_tensor(a, device="cuda"))
            res[f"{k}/act{s}"], res[f"{k}/obs{s}"], res[f"{k}/rew{s}"] = a, obs.cpu().numpy(), rew.cpu().numpy()
            res[f"{k}/term{s}"], res[f"{k}/trunc{s}"] = term.cpu().numpy(), trunc.cpu().numpy()
            res[f"{k}/reset{s}"] = info["reset_idx"].cpu().numpy() if "reset_idx" in info else np.zeros(0, int)
            if "final_obs" in info:
                res[f"{k}/final{s}"] = info["final_obs"].cpu().numpy()
            res[f"{k}/after{s}"] = init_fields(env.handle)
            res[f"{k}/targets_after{s}"] = env._targets.cpu().numpy()
        env.close()

np.savez(out, **res)
"""

# SOFTROD_* settings of a worker process -> the cases it runs
SETTINGS = {"default": ({}, "eq,long,reach,kink,nan,e2e"), "cluster": ({"SOFTROD_LEAN_CLUSTER": "1"}, "eq")}


def _reach_targets():
    """Launch 0: targets of both directions; launch 1: the same with only the last control value of direction 1 changed."""
    tg = _targets(np.random.default_rng(77), LONG_ENVS, 4)
    tg2 = tg.copy()
    tg2[:, 1, 3] = -0.9 * tg[:, 1, 3] + 0.5
    return [tg, tg2]


def _kink(x, Q):
    """In place, on [env, ...] arrays of arms lying along +y with d1 = +z: env e of KINK_AT gets a KINK_DEG kink about
    its d1, the frames of elements KINK_AT[e] .. n-1 turned and the nodes rebuilt along the turned d3."""
    n, t = KINK_N, np.deg2rad(KINK_DEG)
    for e, m in KINK_AT.items():
        ln = np.sqrt(np.sum(np.diff(x[e], axis=1) ** 2, axis=0))
        d1 = Q[e, 0, :, m]
        K = np.array([[0, -d1[2], d1[1]], [d1[2], 0, -d1[0]], [-d1[1], d1[0], 0]])
        R = np.eye(3) + np.sin(t) * K + (1 - np.cos(t)) * (K @ K)
        for k in range(m, n):
            Q[e, :, :, k] = Q[e, :, :, k] @ R.T
            x[e, :, k + 1] = x[e, :, k] + ln[k] * Q[e, 2, :, k]


@pytest.fixture(scope="module")
def worker(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("long_rods_spline")
    script = tmp / "long_rods_spline_worker.py"
    script.write_text(_WORKER)

    @functools.lru_cache(maxsize=None)
    def get(setting):
        extra, cases = SETTINGS[setting]
        env = {k: v for k, v in os.environ.items() if k not in ("SOFTROD_LEAN_CLUSTER", "SOFTROD_FASTPATH", "SOFTROD_LEAN_FOLD")}
        env.update(extra)
        out = tmp / f"{setting}.npz"
        res = subprocess.run([sys.executable, str(script), ROOT, cases, str(out)], stdout=subprocess.PIPE,
                             stderr=subprocess.STDOUT, text=True, env=env, timeout=3000)
        assert res.returncode == 0, res.stdout[-3000:]
        return dict(np.load(out))
    return get


def _oracle(kw, fields0):
    """The C oracle of a case, started from the state the GPU held before the first launch."""
    import rod_oracle as ro
    n = kw["n_elem"]
    r = ro.OracleRod(n, [0, 0, 0], [0, 1.0, 0], [0, 0, 1.0], kw["base_length"], kw["base_radius"], kw["density"],
                     kw["youngs_modulus"], kw["dt"], damping_constant=kw["damping_constant"], bc_kind=kw["bc_kind"],
                     damping_before_constraints=True, spline=kw["spline"])
    parts = np.split(fields0, np.cumsum((3 * (n + 1), 3 * (n + 1), 9 * n, 3 * n))[:-1])
    for name, a in zip(("position_collection", "velocity_collection", "director_collection", "omega_collection"), parts):
        getattr(r, name)[...] = a.reshape(getattr(r, name).shape)
    return r


def _vs_oracle(res, key, name, n, envs, launches, targets, layout):
    """The GPU envs `envs` of case `key` against the C oracle with the same targets before every launch: all eight
    fields within the 1e-9 rule or 20x the oracle's one-ulp divergence (test_long_rods._check_vs_oracle), the tip in the
    observation the float32 cast of the state's, the magnitudes within 1e-9 relative and the cached control values
    equal to the oracle's.  Returns the oracle's magnitudes after every launch, per env."""
    from test_parity_gpu import assert_state_close, one_ulp_divergence, rate_floors
    import rod_oracle as ro
    kw = _arm(name, n)
    dirs, P = kw["spline"]["directions"], kw["spline"]["n_ctrl"]
    mags_out = {}
    for e in envs:
        def mk():
            return _oracle(kw, res[f"{key}/init"][e])

        def advance(rod, refs=None):
            for li, k in enumerate(launches):
                for d in dirs:
                    rod.spline_points[d, :P] = targets[li][e, d]
                rod.substeps(k)
                if refs is not None:
                    refs.append(({f: getattr(rod, f).copy() for f in ORACLE_FIELDS}, rod.spline_points.copy(),
                                 rod.spline_magnitude.copy()))
        rod, refs = mk(), []
        advance(rod, refs)
        rod.close()
        sens = one_ulp_divergence(mk, advance, refs[-1][0])
        for li, (ref, pts, mags) in enumerate(refs):
            what = f"{key} env {e} after launch {li}"
            f = _fields(res[f"{key}/state{li}"][e], layout, n)
            floors = rate_floors(kw["youngs_modulus"], kw["density"], kw["base_length"], n, kw["base_radius"],
                                 np.abs(ref["position_collection"]).max())
            for fname in ORACLE_FIELDS:
                assert_state_close(f[fname], ref[fname], fname, floors, what, measured=sens)
            obs = res[f"{key}/obs{li}"][e]
            np.testing.assert_array_equal(obs[:6], np.float32(np.concatenate([f["position_collection"][:, -1],
                                                                              f["velocity_collection"][:, -1]])))
            for d in dirs:
                np.testing.assert_array_equal(res[f"{key}/pts{li}"][e, d, P:2 * P], pts[d, P:2 * P], err_msg=what)
                np.testing.assert_allclose(res[f"{key}/mags{li}"][e, d], mags[d], rtol=1e-9,
                                           atol=1e-12 * kw["spline"]["scale"], err_msg=what)
        mags_out[e] = [m for _, _, m in refs]
    return mags_out


def _bend_w2(Q, m):
    """The lean kernel's bend-range operand at the Voronoi point between elements m - 1 and m of directors [3, 3, n]
    (rows d1, d2, d3): |axial(R - R^T)|^2 with R = Q_m Q_{m-1}^T."""
    R = Q[:, :, m] @ Q[:, :, m - 1].T
    v = np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]])
    return float(v @ v)


def _launch_targets(seed, n_env, name, launches):
    rng = np.random.default_rng(seed)
    return [_targets(rng, n_env, CASES[name][2]) for _ in launches]


# ---- 1 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", EQ_SIZES)
def test_cluster_spline_kernel_gives_the_bits_of_the_one_cta_kernel(worker, n):
    """SOFTROD_LEAN_CLUSTER=1 (two CTAs per rod, the spline model on clusters) against the default kernel (the spline
    model's one-CTA kernel in 544 / 768 / 1024-thread CTAs): a free arm with directions (0, 1) and no rate limit; a
    clamped arm with directions (0, 1, 2) and a rate limit that keeps the re-fit running through both launches; a clamped
    arm with (0, 1) and that rate limit; new random targets before every launch; 7 envs and 300 envs.  After each of two
    launches (150 and 250 substeps) the whole state block and the spline cache (targets, cached control values, flags
    and magnitudes; a digest of the three per env for the 300-env batches), the observations, rewards and terminated
    flags are equal bit for bit, and no env is terminated."""
    ref, cl = worker("default"), worker("cluster")
    for name in EQ_CASES:
        for size, _ in EQ_BATCHES:
            key = f"eq{n}/{name}/{size}"
            for li in range(len(LAUNCHES)):
                for f in ("state", "obs", "rew", "term") + (("pts", "mags") if size == "small" else ()):
                    a, b = ref[f"{key}/{f}{li}"], cl[f"{key}/{f}{li}"]
                    assert a.shape == b.shape, (key, f)
                    assert np.array_equal(a, b), (key, f, li, np.argwhere(a != b)[:5])
            assert not cl[f"{key}/term{len(LAUNCHES) - 1}"].any(), key
            assert ref[f"{key}/counts"][0] == 0 and cl[f"{key}/counts"][0] == 0, (key, cl[f"{key}/counts"])


# ---- 2 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", LONG_SIZES)
def test_long_spline_rods_vs_c_oracle(worker, n):
    """Arms of 1024-4095 elements (clusters of 3 ... 8 CTAs), two envs per case, against the C oracle started from the
    same state, with the same new random targets before each of two launches (100 and 200 substeps): a free arm with
    directions (0, 1) and no rate limit, and a clamped arm with (0, 1, 2) and a rate limit.  All eight fields within the
    1e-9 rule or 20x the oracle's one-ulp divergence, magnitudes within 1e-9 relative, cached control values equal."""
    res = worker("default")
    for ci, name in enumerate(LONG_CASES):
        key = f"long{n}/{name}"
        _vs_oracle(res, key, name, n, range(LONG_ENVS), LONG_LAUNCHES,
                   _launch_targets(1000 * n + ci, LONG_ENVS, name, LONG_LAUNCHES), res["layout"])
        assert res[f"{key}/counts"][0] == 0 and not res[f"{key}/term{len(LONG_LAUNCHES) - 1}"].any(), key


# ---- 3 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_target_change_reaches_every_rank(worker):
    """n = 2047 (C = 4): after a launch that settles the forcing, a change of only the last control value of direction
    1 re-fits the magnitudes of every element: on the last rank's elements (1536-2046, whose arc lengths continue the
    carry of ranks 0-2) they change and match the oracle's within 1e-9 relative, as do all fields."""
    res = worker("default")
    mags = _vs_oracle(res, "reach", "free01", REACH_N, range(LONG_ENVS), LONG_LAUNCHES, _reach_targets(), res["layout"])
    for e in range(LONG_ENVS):
        before, after = res["reach/mags0"][e, 1, 1536:], res["reach/mags1"][e, 1, 1536:]
        assert np.abs(after - before).min() > 0, e
        np.testing.assert_allclose(after, mags[e][1][1, 1536:], rtol=1e-9, atol=1e-12 * _arm("free01", REACH_N)["spline"]["scale"])


# ---- 4 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_out_of_range_bends_on_clusters(worker):
    """Clamped thin rods of n = 2047 (clusters of 4) with a rate-limited spline, one env kinked by 60 degrees at element
    1200 (inside rank 2), one at elements 511 / 512 (the curvature stencil of Voronoi point 511 reads rank 1's first
    element), stepped one substep per launch for eight launches.  At the kinked Voronoi points the bend stays past the
    spline model's bend map (w2 above twice 0.6144, the operand of the kernel's own range test) before the first
    substep and after every one, so the safe kernel takes its reference map there in every substep; the points next to
    them start straight.  The kinked envs match the C oracle after every substep."""
    res = worker("default")
    n, lay = KINK_N, res["layout"]
    for e, m in KINK_AT.items():
        Q0 = np.split(res["kink/init"][e], np.cumsum((3 * (n + 1), 3 * (n + 1), 9 * n)))[2].reshape(3, 3, n)
        w2 = [_bend_w2(Q0, m)] + [_bend_w2(_fields(res[f"kink/state{li}"][e], lay, n)["director_collection"], m)
                                  for li in range(len(KINK_LAUNCHES))]
        assert min(w2) > 2 * NARROW_BEND_W2, (e, m, w2)
        assert _bend_w2(Q0, m - 1) < 1e-20 and _bend_w2(Q0, m + 1) < 1e-20, e   # (one kinked point per env)
    _vs_oracle(res, "kink", "kink", KINK_N, sorted(KINK_AT), KINK_LAUNCHES,
               _launch_targets(5, KINK_ENVS, "kink", KINK_LAUNCHES), res["layout"])


# ---- 5 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_nan_in_the_last_rank_leaves_the_other_envs_alone(worker):
    """A NaN in the tip's velocity (the last thread of the last CTA) of env 2 terminates env 2 only, and every other
    env's state block, spline cache and observation keep the bits of the same run without the NaN."""
    res = worker("default")
    assert list(res["nan/nan/term"]) == [0, 0, 1, 0] and not res["nan/clean/term"].any(), res["nan/nan/term"]
    for e in (0, 1, 3):
        for f in ("state", "pts", "mags", "obs"):
            assert np.array_equal(res[f"nan/nan/{f}"][e], res[f"nan/clean/{f}"][e]), (e, f)


# ---- 6 -------------------------------------------------------------------------------------------------------------
def _replica_obs(o, target, n):
    """SoftArmTrackingVectorEnv._state of an oracle rod: 4 segment means of kappa[0] and kappa[1], tip, target."""
    from gym_softrobot_b200.envs.soft_arm_tracking import _L, _N_CTRL
    seg = int((n - 1) / _N_CTRL)
    parts = []
    for c in (0, 1):
        k = o.kappa[c]
        m = [k[seg * i:seg * (i + 1)].mean() for i in range(_N_CTRL - 1)] + [k[seg * (_N_CTRL - 1):].mean()]
        parts.append(np.array(m) * _L / (2 * np.pi))
    return np.concatenate([parts[0], parts[1], o.position_collection[:, -1] / _L, target / 1000])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [1, 2])
def test_soft_arm_tracking_2048_elements_vs_c_oracle_replica(worker, mode):
    """gsb.make_vec("SoftArmTracking-v0", 8, n_elems=2048, time_step=5e-6): 2000 substeps per env-step, truncation after
    500 env-steps.  Three env-steps of random actions, envs 1 and 4 brought to the end of their episode in the second
    (truncated and reset inside the same step()).  Against a C-oracle replica of each env (its rod, its spline forcing,
    the env's observation and reward, rebuilt from the reset state after an autoreset): observations, final
    observations and rewards within 1e-9, terminated and truncated flags exact."""
    import rod_oracle as ro
    from gym_softrobot_b200.envs.soft_arm_tracking import _E, _L, _R, spline_scale
    res, k, n = worker("default"), f"e2e{mode}", E2E_N
    assert int(res[f"{k}/update"]) == 2000 and int(res[f"{k}/n_updates"]) == 500
    spl = dict(directions=(0, 1), n_ctrl=4, scale=spline_scale(n), max_rate=INF)
    kw = dict(n_elem=n, dt=E2E_DT, base_length=_L, base_radius=_R, density=1e-3, youngs_modulus=_E,
              damping_constant=_E * 1e-7, bc_kind=BC_ONE_END_FIXED, spline=spl)
    rods = [_oracle(kw, res[f"{k}/init"][e]) for e in range(E2E_ENVS)]
    tick = np.zeros(E2E_ENVS, int)
    targets = res[f"{k}/targets0"]
    for e in range(E2E_ENVS):
        np.testing.assert_allclose(res[f"{k}/obs_reset"][e], _replica_obs(rods[e], targets[e, 0], n), rtol=1e-9, atol=1e-9)
    for s in range(E2E_STEPS):
        tick[:] = res[f"{k}/tick{s}"]
        a = res[f"{k}/act{s}"]
        for e, o in enumerate(rods):
            o.spline_points[0, :4], o.spline_points[1, :4] = a[e, :4], a[e, 4:]
        ro.substeps_batch(rods, 2000)
        tick += 1
        reset = set(res[f"{k}/reset{s}"].tolist())
        assert reset == (set(E2E_RESET) if s == 1 else set()), (s, reset)
        np.testing.assert_array_equal(res[f"{k}/trunc{s}"], [e in reset for e in range(E2E_ENVS)])
        assert not res[f"{k}/term{s}"].any(), s
        for e, o in enumerate(rods):
            ob = _replica_obs(o, targets[e, min(tick[e], 500)], n)
            tip = o.position_collection[:, -1]
            rew = -np.sum(((targets[e, min(tick[e], 500)] - tip) / 1000) ** 2)
            np.testing.assert_allclose(res[f"{k}/rew{s}"][e], rew, rtol=1e-9, atol=1e-9, err_msg=f"step {s} env {e}")
            if e in reset:
                i = list(res[f"{k}/reset{s}"]).index(e)
                np.testing.assert_allclose(res[f"{k}/final{s}"][i], ob, rtol=1e-9, atol=1e-9, err_msg=f"step {s} env {e}")
            else:
                np.testing.assert_allclose(res[f"{k}/obs{s}"][e], ob, rtol=1e-9, atol=1e-9, err_msg=f"step {s} env {e}")
        targets = res[f"{k}/targets_after{s}"]
        for e in reset:     # the reset env's replica restarts from the state the GPU reset it to
            rods[e].close()
            rods[e] = _oracle(kw, res[f"{k}/after{s}"][e])
            tick[e] = 0
            np.testing.assert_allclose(res[f"{k}/obs{s}"][e], _replica_obs(rods[e], targets[e, 0], n), rtol=1e-9, atol=1e-9)
    for o in rods:
        o.close()
