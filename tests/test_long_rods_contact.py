"""Rods on the frictional plane of 512-4095 elements on thread-block clusters (the plane and muscle models in the
cluster layout of rod_kernel_lean.cuh, DESIGN.md §4.2): plane contact with anisotropic friction, per-env rest curvature
and the travelling-wave muscle.

One rod spans C = ceil((n + 1) / 512) CTAs of a cluster, and the substep is the plane / muscle model's: the cluster
kernel must give the bits of the one-CTA kernels where both exist (SOFTROD_LEAN_CLUSTER=1 forces it for 512-1023
elements), and match the C oracle above 1023 elements, where it is the only kernel.

CPU: sr_create admits 1024-4095 elements for the rod on the plane and / or with the muscle wave, and rejects that model
combined with anything the cluster layout does not build; the C oracle steps such rods.
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

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BC_FREE, BC_ONE_END_FIXED, BC_PENDULUM_SLIDER = 0, 1, 2     # (= _native / rod_oracle)
LONG_3D = "SR_MODEL_SOFT_PENDULUM_3D with SR_BC_MOVING_BASE and laplace_filter_order = 7"

EQ_SIZES = (512, 513, 600, 767, 1000, 1023)   # 512: the tip node alone in rank 1; 1023: both CTAs full
EQ_BATCHES = (("small", 7), ("big", 300))      # 300 envs: more clusters than are resident at once
EQ_MODELS = ("cfirst", "tilted", "snake")
LAUNCHES = (400, 600)
BOUNDARY = (508, 517)                          # elements that must lie on the plane: both sides of rank 0 / 1
LONG_SIZES = (1024, 1535, 2047, 2048, 3000, 4095)   # C = 3 ... 8, last CTA holding 1 ... 512 threads
LONG_CASES = ("cfirst", "ffirst", "muscle")
LONG_ENVS = 2
REACH_N, REACH_FROM = 2047, 1024               # rest curvature only on the Voronoi points of ranks 2 and 3
KINK_N, KINK_ENVS, KINK_DEEP, KINK_EDGE = 2047, 5, 1, 3
KINK_AT = {KINK_DEEP: 1200, KINK_EDGE: 512}    # first element turned: inside rank 2 / rank 1's first (Voronoi 511)
KINK_DEG = 60.0     # past the plane models' 37-degree bend map for all 12 substeps
KINK_LAUNCHES = (3, 3, 3, 3)                   # (the pair stays on: the fallback counters are first polled at step 8)
R0 = 0.004
TILTED = (0.3, -0.2, 1.0)


def _unit(v):
    v = np.asarray(v, float)
    return v / np.linalg.norm(v)


def _frame(normal):
    """(N, a, b): the unit plane normal, the rod's axis in the plane, the second in-plane direction."""
    N = _unit(normal)
    a = _unit(np.cross(N, [1.0, 0.0, 0.0]) if abs(N[0]) < 0.9 else np.cross(N, [0.0, 1.0, 0.0]))
    return N, a, np.cross(N, a)


def _contact(normal, before_forcing, mu=1.0):
    """OctoArmSingle's plane and friction (arm_contact_params), the plane through -R0 N: a rod along the plane through the
    origin rests on it."""
    from gym_softrobot_b200.envs.arm_single import arm_contact_params
    c = arm_contact_params(friction_multiplier=mu, before_forcing=before_forcing)
    N = _unit(normal)
    c["plane_origin"], c["plane_normal"] = list(-R0 * N), list(N)
    return c


def _muscle(normal):
    """ContinuumSnake's MuscleTorques about the plane normal (in-plane undulation), ramped up within the first 0.5 ms."""
    return dict(period=1.0, ramp_up_time=5e-4, phase_shift=0.7, direction=list(_unit(normal)))


def _case(name, n):
    """Handle / oracle keyword arguments of a named case: test_long_rods' rod (L = 1 m, r = 4 mm, dt = 2e-6 x 1023 / n)."""
    normal, bc, before, mu, mus = (0.0, 0.0, 1.0), BC_FREE, False, 1.0, False
    if name == "cfirst":
        before = True
    elif name == "tilted":
        normal, bc = TILTED, BC_ONE_END_FIXED
    elif name == "ffirst":
        bc = BC_ONE_END_FIXED
    elif name == "snake":
        normal, mus = (0.0, 1.0, 0.0), True
    elif name == "muscle":
        normal, mu, mus = (0.0, 1.0, 0.0), 0.0, True
    N, a, b = _frame(normal)
    kw = dict(n_elem=n, dt=2e-6 * 1023 / n, base_length=1.0, base_radius=R0, density=1000.0, youngs_modulus=1e6,
              gravity=tuple(-9.81 * N + (1.5 * b if name == "tilted" else 0.0)), damping_constant=1e-2, bc_kind=bc,
              contact=_contact(normal, before, mu))
    if mus:
        kw["muscle"] = _muscle(normal)
    return kw, N, a


def _init(N, a, n_env):
    """sr_reset rows: every rod starts at the origin along a, its d1 along the plane normal."""
    return np.tile(np.concatenate([np.zeros(3), a, N]), (n_env, 1))


def _rest_kappa(rng, n_env, n, lo=0):
    """Smooth random rest curvature about d1 (in the plane), [n_env, 3, n - 1], zero on the Voronoi points below lo."""
    s = np.linspace(0.0, 1.0, n - 1)
    rk = np.zeros((n_env, 3, n - 1))
    for e in range(n_env):
        for k in range(1, 4):
            rk[e, 0] += rng.uniform(-3.0, 3.0) * np.sin(np.pi * k * s + rng.uniform(0, np.pi))
    rk[:, :, :lo] = 0.0
    return rk


def _wave(rng, n_env, n):
    """Random muscle wave: [n_env] wave numbers and [n_env, n] beta(s) profiles."""
    s = np.linspace(0.0, 1.0, n)
    kw = rng.uniform(3.0, 12.0, n_env)
    beta = np.stack([rng.uniform(-2e-4, 2e-4) * np.sin(np.pi * s) + rng.uniform(-1e-4, 1e-4) * np.sin(3 * np.pi * s)
                     for _ in range(n_env)])
    return kw, beta


# ---- CPU -----------------------------------------------------------------------------------------------------------
def _cfg(n, **kw):
    """A free rod of n elements on a +z plane; keyword arguments set SrConfig fields (lists for the array fields)."""
    from gym_softrobot_b200 import _native as nat
    cfg = nat.SrConfig()
    cfg.struct_size = C.sizeof(nat.SrConfig)
    cfg.model, cfg.n_env, cfg.n_elem, cfg.bc_kind = nat.MODEL_ROD, 4, n, nat.BC_FREE
    cfg.dt, cfg.base_length, cfg.base_radius, cfg.density, cfg.youngs_modulus = 1e-6, 1.0, R0, 1000.0, 1e6
    cfg.damping_constant = 1e-2
    cfg.contact_on, cfg.slip_velocity_tol, cfg.contact_k, cfg.contact_nu = 1, 1e-8, 1e2, 1e1
    cfg.plane_normal[:] = [0.0, 0.0, 1.0]
    cfg.plane_origin[:] = [0.0, 0.0, -R0]
    for k, v in kw.items():
        if isinstance(v, (list, tuple)):
            getattr(cfg, k)[:] = list(v)
        else:
            setattr(cfg, k, v)
    return cfg


MUSCLE_ON = dict(muscle_on=1, muscle_period=1.0, muscle_ramp_up_time=1.0)


@pytest.mark.parametrize("n", [2048, 4095])
@pytest.mark.parametrize("kw", [
    dict(),
    dict(bc_kind=BC_ONE_END_FIXED),
    dict(plane_normal=list(TILTED)),
    dict(contact_on=0, **MUSCLE_ON),
    dict(**MUSCLE_ON),
], ids=["free", "clamped", "tilted", "muscle", "contact-muscle"])
def test_create_accepts_long_rods_on_the_plane(kw, n):
    """The rod on the plane and / or with the muscle wave passes every argument check at 2048 and 4095 elements: no GPU,
    the device error; a B200, a handle."""
    from gym_softrobot_b200 import _native as nat
    lib = nat.load_library()
    h = C.c_void_p()
    rc = lib.sr_create(C.byref(_cfg(n, **kw)), C.byref(h))
    assert rc in (0, -3), lib.sr_last_error().decode()
    if rc == 0:
        lib.sr_destroy(h)


@pytest.mark.parametrize("kw", [
    dict(bc_kind=BC_PENDULUM_SLIDER),
    dict(point_force_on_base=1),
    dict(dtype=1),
    dict(math=1),
    dict(tip_radius=0.002),
    dict(n_rod_per_env=2),
    dict(sucker_on=1, sucker_index=0),
    dict(spline_dir_mask=1, spline_n_ctrl=4, spline_max_rate=1.0),
    dict(laplace_filter_order=7),
], ids=["slider", "point-force", "fp32", "faithful", "tapered", "assembly", "sucker", "spline", "laplace"])
def test_create_rejects_long_contact_rods_it_does_not_build(kw):
    """Checked ahead of the device check, with the message that names what is built: the same answer with or without
    a GPU."""
    from gym_softrobot_b200 import _native as nat
    lib = nat.load_library()
    h = C.c_void_p()
    rc = lib.sr_create(C.byref(_cfg(2048, **kw)), C.byref(h))
    assert rc == -1 and not h.value
    msg = lib.sr_last_error().decode()
    assert msg.startswith("sr_create: " + LONG_ONLY) and LONG_3D in msg, msg


def test_oracle_steps_long_rods_on_the_plane():
    """The C oracle (the GPU tests' reference) steps a 2048-element rod on the plane with rest curvature, and one with
    the muscle wave: finite, and still lying on the plane."""
    import rod_oracle as ro
    n = 2048
    for name in ("ffirst", "snake"):
        kw, N, a = _case(name, n)
        r = ro.OracleRod(n, np.zeros(3), a, N, kw["base_length"], R0, kw["density"], kw["youngs_modulus"], kw["dt"],
                         gravity=kw["gravity"], damping_constant=kw["damping_constant"], bc_kind=kw["bc_kind"],
                         contact=kw["contact"], muscle=kw.get("muscle"))
        r.rest_kappa[...] = _rest_kappa(np.random.default_rng(1), 1, n)[0]
        if "muscle" in kw:
            kwv, beta = _wave(np.random.default_rng(2), 1, n)
            r.muscle[0] = kwv[0]; r.muscle[1:] = beta[0]
        r.substeps(200)
        x = r.position_collection
        assert np.isfinite(x).all() and np.isfinite(r.velocity_collection).all(), name
        assert np.abs(r.velocity_collection).max() > 0, name
        gap = N @ (0.5 * (x[:, :-1] + x[:, 1:])) + R0 - R0 / np.sqrt(r.dilatation)   # (surface_tol = 1e-4)
        assert gap.max() <= 1e-4, (name, gap.max())
        r.close()


# ---- the GPU worker --------------------------------------------------------------------------------------------------
_WORKER = r"""
import hashlib, os, sys
import numpy as np
root, cases, out = sys.argv[1], sys.argv[2].split(","), sys.argv[3]
sys.path[:0] = [root, os.path.join(root, "tests")]
import torch
import test_long_rods_contact as tc
from gym_softrobot_b200 import _native as nat
res = {}

def counts(h):
    return np.array([h.fallback_count(), *h.fallback_causes(), h.launch_count])

def init_fields(h):
    return np.concatenate([h.fields()[k].cpu().numpy().reshape(h.n_env, -1) for k in
                           ("position_collection", "velocity_collection", "director_collection", "omega_collection")], axis=1)

def layout(h):
    return np.array([getattr(h.state_view(), f) for f in ("f_position", "f_velocity", "f_director", "f_omega",
                                                           "f_tangents", "f_kappa", "f_sigma", "f_dilatation")])

def make(name, n, n_env, rng, lo=0):
    kw, N, a = tc._case(name, n)
    h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, math=nat.MATH_FAST, **kw)
    h.reset_host(tc._init(N, a, n_env))
    rk = tc._rest_kappa(rng, n_env, n, lo)
    h.rest_kappa_tensor()[:] = torch.as_tensor(rk, device="cuda")
    wave = None
    if "muscle" in kw:
        wave = tc._wave(rng, n_env, n)
        mu = h.muscle_tensor()
        mu[:, 1] = torch.as_tensor(wave[0], device="cuda")
        mu[:, 2:] = torch.as_tensor(wave[1], device="cuda")
    torch.cuda.synchronize()
    return h, rk, wave

def run(key, h, launches, rng, full, new_kappa=False):
    for li, k in enumerate(launches):
        if new_kappa and li > 0:   # a fresh random rest curvature before every launch
            h.rest_kappa_tensor()[:] = torch.as_tensor(tc._rest_kappa(rng, h.n_env, h.n_elem), device="cuda")
            torch.cuda.synchronize()
        o, r, t = h.step_host(None, k)
        res[f"{key}/obs{li}"], res[f"{key}/rew{li}"], res[f"{key}/term{li}"] = o.copy(), r.copy(), t.copy()
        st = h.state_tensor().cpu().numpy()
        assert np.isfinite(st).all(), key
        res[f"{key}/state{li}"] = st if full else np.array([hashlib.blake2b(e.tobytes(), digest_size=16).digest() for e in st])
        if li == 0 and not full:
            res[f"{key}/state0_env0"] = st[0]
    res[f"{key}/counts"] = counts(h)

def set_fields(h, **arrays):
    fl = h.fields()
    for k, a in arrays.items():
        fl[k][:] = torch.as_tensor(a, device="cuda")
    torch.cuda.synchronize()     # (the handle steps on a stream of its own)

for n in (tc.EQ_SIZES if "eq" in cases else (512,) if "eq512" in cases else ()):
    for size, n_env in tc.EQ_BATCHES:
        for mi, name in enumerate(tc.EQ_MODELS):
            rng = np.random.default_rng(100 * n + n_env + mi)
            h, _, _ = make(name, n, n_env, rng)
            res["layout"] = layout(h)
            run(f"eq{n}/{name}/{size}", h, tc.LAUNCHES, rng, size == "small", new_kappa=True)
            h.close()

if "long" in cases:
    for n in tc.LONG_SIZES:
        for ci, name in enumerate(tc.LONG_CASES):
            h, rk, wave = make(name, n, tc.LONG_ENVS, np.random.default_rng(1000 * n + ci))
            res[f"long{n}/{name}/init"] = init_fields(h)
            run(f"long{n}/{name}", h, tc.LAUNCHES, None, True)
            if wave is not None:
                res[f"long{n}/{name}/clock"] = h.muscle_tensor()[:, 0].cpu().numpy()
            res["layout"] = layout(h)
            h.close()

if "reach" in cases:
    h, rk, _ = make("cfirst", tc.REACH_N, tc.LONG_ENVS, np.random.default_rng(77), lo=tc.REACH_FROM)
    res["reach/init"] = init_fields(h)
    run("reach", h, tc.LAUNCHES, None, True)
    res["layout"] = layout(h)
    h.close()

if "kink" in cases:
    h, rk, _ = make("ffirst", tc.KINK_N, tc.KINK_ENVS, np.random.default_rng(5))
    fl = h.fields()
    x, Q = (fl[k].cpu().numpy() for k in ("position_collection", "director_collection"))
    tc._kink(x, Q)
    set_fields(h, position_collection=x, director_collection=Q)
    res["kink/init"] = init_fields(h)
    run("kink", h, tc.KINK_LAUNCHES, None, True)
    res["layout"] = layout(h)
    h.close()

if "nan" in cases:
    h, _, _ = make("snake", 2047, 4, np.random.default_rng(9))
    v = h.fields()["velocity_collection"].cpu().numpy()
    v[2, 1, h.n_elem] = np.nan          # the tip node: the last thread of the last rank
    set_fields(h, velocity_collection=v)
    o, r, t = h.step_host(None, 20)
    res["nan/term"], res["nan/rew"] = t.copy(), r.copy()
    h.close()

np.savez(out, **res)
"""

# SOFTROD_* settings of a worker process -> the cases it runs
SETTINGS = {"default": ({}, "eq,long,reach,kink,nan"), "cluster": ({"SOFTROD_LEAN_CLUSTER": "1"}, "eq"),
            "safe": ({"SOFTROD_FASTPATH": "0"}, "kink"), "nofold": ({"SOFTROD_LEAN_FOLD": "0"}, "eq512")}


def _kink(x, Q):
    """In place, on [env, ...] arrays of rods lying along the plane: env KINK_DEEP and env KINK_EDGE get a KINK_DEG kink
    in the plane, the frames of elements KINK_AT[e] .. n-1 turned about their d1 (the plane normal) and the nodes rebuilt
    along the turned d3."""
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
    tmp = tmp_path_factory.mktemp("long_rods_contact")
    script = tmp / "long_rods_contact_worker.py"
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


def _gaps(st, layout, n, normal):
    """Per element: height of the element's centre above the plane minus its current radius (the kernel's contact gap,
    up to the half step by which the stored dilatation lags the positions)."""
    N = _unit(normal)
    p, dl = layout[0], layout[7]
    x = st[p:p + 3, :n + 1]
    return N @ (0.5 * (x[:, :-1] + x[:, 1:])) + R0 - R0 / np.sqrt(st[dl, :n])


def _oracle_factory(kw, init_row, fields0, rk, wave):
    import rod_oracle as ro
    n = kw["n_elem"]

    def mk():
        r = ro.OracleRod(n, init_row[0:3], init_row[3:6], init_row[6:9], kw["base_length"], kw["base_radius"],
                         kw["density"], kw["youngs_modulus"], kw["dt"], gravity=kw["gravity"],
                         damping_constant=kw["damping_constant"], bc_kind=kw["bc_kind"], contact=kw["contact"],
                         muscle=kw.get("muscle"))
        parts = np.split(fields0, np.cumsum((3 * (n + 1), 3 * (n + 1), 9 * n, 3 * n))[:-1])
        for name, a in zip(("position_collection", "velocity_collection", "director_collection", "omega_collection"), parts):
            getattr(r, name)[...] = a.reshape(getattr(r, name).shape)
        r.rest_kappa[...] = rk
        if wave is not None:
            r.muscle[0] = wave[0]; r.muscle[1:] = wave[1]
        return r
    return mk


def _vs_oracle(res, key, name, n, envs, launches, rng_seed, lo=0, kinked=False):
    """The GPU envs `envs` of case `key` against the C oracle started from the state the GPU held before the first launch,
    with the same rest curvature and muscle wave: all eight fields and the tip in the observation after every launch,
    within the 1e-9 rule or 20x the oracle's one-ulp divergence (test_long_rods._check_vs_oracle)."""
    kw, N, a = _case(name, n)
    rng = np.random.default_rng(rng_seed)
    n_env = KINK_ENVS if kinked else LONG_ENVS
    rk = _rest_kappa(rng, n_env, n, lo)
    wave = _wave(rng, n_env, n) if "muscle" in kw else None
    init = _init(N, a, n_env)
    from test_parity_gpu import assert_state_close, one_ulp_divergence, rate_floors
    import rod_oracle as ro
    layout = res["layout"]
    mks = [_oracle_factory(kw, init[e], res[f"{key}/init"][e], rk[e], None if wave is None else (wave[0][e], wave[1][e]))
           for e in envs]
    rods, refs = [mk() for mk in mks], [[] for _ in envs]
    for k in launches:
        ro.substeps_batch(rods, k)
        for i, o in enumerate(rods):
            refs[i].append({f: getattr(o, f).copy() for f in ORACLE_FIELDS})
    for o in rods:
        o.close()
    for i, e in enumerate(envs):
        # the oracle's one-ulp divergence over the whole horizon (measured per env, used at every launch)
        sens = one_ulp_divergence(mks[i], lambda rod: rod.substeps(sum(launches)), refs[i][-1])
        for li, ref in enumerate(refs[i]):
            f = _fields(res[f"{key}/state{li}"][e], layout, n)
            x = ref["position_collection"]
            floors = rate_floors(kw["youngs_modulus"], kw["density"], kw["base_length"], n, R0, np.abs(x).max())
            for fname in ORACLE_FIELDS:
                assert_state_close(f[fname], ref[fname], fname, floors, f"{key} env {e} after launch {li}", measured=sens)
            # the tip in the observation: the float32 cast of the state block's tip, which the rule above has checked;
            # against the oracle within 2 float32 ulp, or 20x the oracle's one-ulp divergence as for the state
            obs = res[f"{key}/obs{li}"][e]
            np.testing.assert_array_equal(obs[:6], np.float32(np.concatenate([f["position_collection"][:, -1],
                                                                              f["velocity_collection"][:, -1]])))
            for sl, fname in ((slice(0, 3), "position_collection"), (slice(3, 6), "velocity_collection")):
                np.testing.assert_allclose(obs[sl], ref[fname][:, -1], rtol=2e-6, atol=max(1e-7, 20.0 * sens[fname]))


# ---- 1 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", EQ_SIZES)
def test_cluster_contact_kernel_gives_the_bits_of_the_one_cta_kernels(worker, n):
    """SOFTROD_LEAN_CLUSTER=1 (two CTAs per rod, the plane / muscle model on clusters) against the default kernels (the
    CTA layout in 544 / 768 / 1024-thread CTAs; at n = 512 the reference is the plane model's 544-thread kernel,
    SOFTROD_LEAN_FOLD=0, since its fold layout differs in the padding slots; the muscle model has no fold layout): a free rod on a +z
    plane, contact first; a clamped rod on a tilted plane under a gravity that drags it sideways, forcing first; a free rod on
    a +y plane with the travelling-wave muscle (random beta(s) and wave number), forcing first; a fresh random rest
    curvature before every launch; 7 envs and 300 envs.  After each of two launches (400 and 600 substeps) the whole
    state block (a digest per env for the 300-env batches), the observations, rewards and terminated flags are equal
    bit for bit, with no range fallback; after the first launch elements 508-516 lie on the plane, so that the contact
    loads cross the rank boundary."""
    ref, cl = worker("nofold" if n == 512 else "default"), worker("cluster")
    for mi, name in enumerate(EQ_MODELS):
        normal = _case(name, n)[1]
        for size, _ in EQ_BATCHES:
            key = f"eq{n}/{name}/{size}"
            for li in range(len(LAUNCHES)):
                for f in ("state", "obs", "rew", "term"):
                    a, b = ref[f"{key}/{f}{li}"], cl[f"{key}/{f}{li}"]
                    assert a.shape == b.shape, (key, f)
                    assert np.array_equal(a, b), (key, f, li, np.argwhere(a != b)[:5])
            assert ref[f"{key}/counts"][0] == 0 and cl[f"{key}/counts"][0] == 0, (key, cl[f"{key}/counts"])
            assert not cl[f"{key}/term{len(LAUNCHES) - 1}"].any()
            st = cl[f"{key}/state0"][0] if size == "small" else cl[f"{key}/state0_env0"]
            gap = _gaps(st, cl["layout"], n, normal)[BOUNDARY[0]:min(BOUNDARY[1], n)]
            assert (gap <= 1e-4).all(), (key, gap)


# ---- 2 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", LONG_SIZES)
def test_long_contact_rods_vs_c_oracle(worker, n):
    """Rods on the plane of 1024-4095 elements (clusters of 3 ... 8 CTAs), two envs per case, against the C oracle
    started from the same state, after 400 and 1000 substeps: a free rod with rest curvature, contact first (round-off
    limited); a clamped rod with rest curvature from rest, forcing first (the regularised stick-slip chatters: the
    oracle's measured one-ulp divergence is the floor); the muscle wave on a frictionless +y plane.  All eight fields
    within the 1e-9 rule or 20x the oracle's one-ulp divergence; the tip in the observation equal to the float32 cast
    of the state's tip and within the same measured floor of the oracle's; the muscle clock is the oracle's time."""
    res = worker("default")
    for ci, name in enumerate(LONG_CASES):
        key = f"long{n}/{name}"
        _vs_oracle(res, key, name, n, range(LONG_ENVS), LAUNCHES, 1000 * n + ci)
        cnt = res[f"{key}/counts"]
        assert cnt[0] == 0, (key, cnt)
        if name == "muscle":
            t = sum(LAUNCHES) * _case(name, n)[0]["dt"]
            np.testing.assert_allclose(res[f"{key}/clock"], t, rtol=1e-12)


# ---- 3 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_actuation_reaches_every_rank(worker):
    """Rest curvature on the Voronoi points of ranks 2 and 3 only (n = 2047, j >= 1024) moves the rod as it moves the
    oracle's: every field within the 1e-9 rule or 20x the oracle's one-ulp divergence, and the actuated part moves in
    the plane (across the rod's axis: gravity and the plane's response act along the normal)."""
    res = worker("default")
    _vs_oracle(res, "reach", "cfirst", REACH_N, range(LONG_ENVS), LAUNCHES, 77, lo=REACH_FROM)
    _, N, a = _case("cfirst", REACH_N)
    lay = res["layout"]
    v = res[f"reach/state{len(LAUNCHES) - 1}"][:, lay[1]:lay[1] + 3, :REACH_N + 1]
    across = np.abs(np.einsum("i,eik->ek", np.cross(N, a), v))
    assert (across[:, REACH_FROM:].max(1) > 1e-6).all(), across.max(1)


# ---- 4 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_contact_range_fallback_across_ctas(worker):
    """Clamped rods of n = 2047 on the plane (clusters of 4), one env kinked in the plane by 60 degrees at element 1200
    (inside rank 2), one at elements 511 / 512 (the curvature stencil of Voronoi point 511 reads rank 1's first element).
    The fast-only kernel flags both envs in every launch, with cause "bend" only; the state block, observations, rewards
    and flags equal the safe kernel's alone (SOFTROD_FASTPATH=0) bit for bit after every launch, and the kinked envs
    match the C oracle."""
    res, safe = worker("default"), worker("safe")
    L = len(KINK_LAUNCHES)
    for li in range(L):
        for f in ("state", "obs", "rew", "term"):
            a, b = res[f"kink/{f}{li}"], safe[f"kink/{f}{li}"]
            assert np.array_equal(a, b), (f, li, np.argwhere(a != b)[:5])
    cnt = res["kink/counts"]
    assert list(cnt[:4]) == [2 * L, 0, 2 * L, 0], cnt                 # total, rotation, bend, stretch
    assert cnt[4] == 1 + 2 * L and safe["kink/counts"][4] == 1 + L, (cnt, safe["kink/counts"])
    _vs_oracle(res, "kink", "ffirst", KINK_N, sorted(KINK_AT), KINK_LAUNCHES, 5, kinked=True)


# ---- 5 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_nan_in_the_last_rank_terminates_that_env_only(worker):
    """A NaN in the tip's velocity (the last thread of the last CTA) of a muscle-driven rod on the plane reaches rank
    0's lead through the cluster's NaN flag: env 2 is terminated and no other env."""
    res = worker("default")
    assert list(res["nan/term"]) == [0, 0, 1, 0], res["nan/term"]
