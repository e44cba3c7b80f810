"""Rods of 512-4095 elements on thread-block clusters (the plain model in the cluster layout of rod_kernel_lean.cuh,
DESIGN.md §4.2).

One rod spans C = ceil((n + 1) / 512) CTAs of a cluster, and the substep is the plain model's: the cluster kernel must
give the bits of the one-CTA kernels where both exist (SOFTROD_LEAN_CLUSTER=1 forces it for 512-1023 elements), and
match the C oracle above 1023 elements, where it is the only kernel.

CPU: sr_create admits 1024-4095 elements for the plain model only, with a message naming what is built; the C oracle
steps such rods.
GPU: each kernel setting runs in a subprocess of its own (the settings are read once per process), and the saved
outputs are compared: the forced cluster kernel against the default kernels, the default (cluster) pair against the
safe kernel alone (SOFTROD_FASTPATH=0) and the C oracle."""
import ctypes as C
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BC_FREE, BC_ONE_END_FIXED, BC_PENDULUM_SLIDER = 0, 1, 2     # (= _native / rod_oracle)

EQ_SIZES = (512, 513, 600, 767, 1000, 1023)   # 512: the tip node alone in rank 1; 1023: both CTAs full
EQ_BATCHES = (("small", 7), ("big", 300))      # 300 envs: more clusters than are resident at once
LAUNCHES = (400, 600)
LONG_SIZES = (1024, 1535, 2047, 2048, 3000, 4095)   # C = 3 ... 8, last CTA holding 1 ... 512 threads
LONG_BCS = (BC_FREE, BC_ONE_END_FIXED, BC_PENDULUM_SLIDER)
KINK_N, KINK_ENVS, KINK_DEEP, KINK_EDGE = 2047, 5, 1, 3
KINK_AT = {KINK_DEEP: 1200, KINK_EDGE: 512}    # first element turned: inside rank 2 / rank 1's first (Voronoi 511)
KINK_DEG = 45.0     # past the bend map's range (4 sin^2 = 0.6144: 23 degrees) for all 12 substeps; a 30-degree kink of
                    # these fine elements springs back below it within ~12 substeps
KINK_LAUNCHES = (3, 3, 3, 3)                   # (the pair stays on: the fallback counters are first polled at step 8)
ORACLE_FIELDS = ("position_collection", "velocity_collection", "director_collection", "omega_collection",
                 "tangents", "kappa", "sigma", "dilatation")


def _rod_cfg(n, bc, damper=True, gravity=(0.0, -9.80665, 0.0)):
    """test_generic_rod_vs_oracle's n = 1023 rod (r = 4 mm, dt = 2e-6), with dt scaled by 1023 / n."""
    return dict(n_elem=n, dt=2e-6 * 1023 / n, base_length=1.0, base_radius=0.004, density=1000.0, youngs_modulus=1e6,
                gravity=gravity, damping_constant=2e-3 if damper else -1.0, bc_kind=bc)


def _eq_cfg(n, bc):
    """Equality cases: gravity with all three components non-zero, the damper on for every other BC."""
    rng = np.random.default_rng(n + 10 * bc)
    g = rng.uniform(1.0, 3.0, 3) * rng.choice([-1.0, 1.0], 3)
    return _rod_cfg(n, bc, damper=bc != BC_FREE, gravity=tuple(9.80665 * g / np.linalg.norm(g)))


def _random_init(rng, n_env):
    """sr_reset rows: random start, random direction, a random normal perpendicular to it."""
    init = np.zeros((n_env, 9))
    for e in range(n_env):
        d = rng.normal(size=3); d /= np.linalg.norm(d)
        m = np.cross(d, rng.normal(size=3)); m /= np.linalg.norm(m)
        init[e] = [*rng.uniform(-1, 1, 3), *d, *m]
    return init


def _pendulum_dt(n):
    return 2e-6 * 1023 / n


# ---- CPU -----------------------------------------------------------------------------------------------------------
def _cfg(**kw):
    from gym_softrobot_b200 import _native as nat
    cfg = nat.SrConfig()
    cfg.struct_size = C.sizeof(nat.SrConfig)
    cfg.model, cfg.n_env, cfg.n_elem, cfg.bc_kind = nat.MODEL_SOFT_PENDULUM, 4, 2048, nat.BC_PENDULUM_SLIDER
    cfg.point_force_on_base = 1
    cfg.dt, cfg.base_length, cfg.base_radius, cfg.density, cfg.youngs_modulus = 5e-6, 1.0, 0.05, 1000.0, 1e6
    cfg.damping_constant = 2e-3
    for k, v in kw.items():
        setattr(cfg, k, v)
    return cfg


LONG_ONLY = "n_elem of 1024-4095 is built for SR_DTYPE_F64, SR_MATH_FAST, SR_MODEL_ROD or SR_MODEL_SOFT_PENDULUM"


@pytest.mark.parametrize("kw,msg", [
    (dict(n_elem=4096), "n_elem <= 4095"),
    (dict(dtype=1), LONG_ONLY),                                   # FP32 storage
    (dict(math=1), LONG_ONLY),                                    # faithful math
    (dict(model=2, bc_kind=3, base_move_period=0.04), LONG_ONLY),   # SoftPendulum3D (moving base)
    (dict(contact_on=1, slip_velocity_tol=1e-4), LONG_ONLY),
    (dict(model=0, bc_kind=0, point_force_on_base=0, n_rod_per_env=2), LONG_ONLY),
], ids=["4096", "fp32", "faithful", "pendulum3d", "contact", "two_rods"])
def test_create_rejects_long_rods_it_does_not_build(kw, msg):
    """Checked with the other arguments, ahead of the device check: the same answer with or without a GPU."""
    from gym_softrobot_b200 import _native as nat
    lib = nat.load_library()
    h = C.c_void_p()
    rc = lib.sr_create(C.byref(_cfg(**kw)), C.byref(h))
    assert rc == -1 and not h.value
    assert msg in lib.sr_last_error().decode()


@pytest.mark.parametrize("kw", [dict(), dict(model=0, bc_kind=1, point_force_on_base=0, n_elem=4095)], ids=["pendulum", "rod"])
def test_create_accepts_long_rods_it_builds(kw):
    """SoftPendulum-v0's model at n = 2048 and a clamped rod at n = 4095 pass every argument check: no GPU, the device
    error; a B200, a handle."""
    from gym_softrobot_b200 import _native as nat
    lib = nat.load_library()
    h = C.c_void_p()
    rc = lib.sr_create(C.byref(_cfg(**kw)), C.byref(h))
    assert rc in (0, -3), lib.sr_last_error().decode()
    if rc == 0:
        lib.sr_destroy(h)


def test_oracle_steps_long_rods():
    """The C oracle steps an n = 4095 clamped rod and SoftPendulum-v0 at n_elems = 2048 (the GPU tests' reference)."""
    import rod_oracle as ro
    r = ro.OracleRod(4095, np.zeros(3), [1.0, 0.0, 0.0], [0.0, 1.0, 0.0], 1.0, 0.004, 1000.0, 1e6, 2e-6 * 1023 / 4095,
                     gravity=(0.0, -9.80665, 0.0), damping_constant=2e-3, bc_kind=ro.BC_ONE_END_FIXED)
    r.substeps(200)
    assert np.isfinite(r.position_collection).all() and np.abs(r.velocity_collection).max() > 0
    r.close()
    e = ro.OracleSoftPendulum(n_elems=2048, time_step=_pendulum_dt(2048), recording_fps=2500)
    e.reset(seed=3)
    obs, rew, term, trunc, _ = e.step(np.float32(15.0))
    assert np.isfinite(obs).all() and not term and not trunc and np.isfinite(rew)


# ---- the GPU worker --------------------------------------------------------------------------------------------------
_WORKER = r"""
import hashlib, os, sys
import numpy as np
root, cases, out = sys.argv[1], sys.argv[2].split(","), sys.argv[3]
sys.path[:0] = [root, os.path.join(root, "tests")]
import torch
import test_long_rods as tl
from gym_softrobot_b200 import _native as nat
from gym_softrobot_b200.envs.soft_pendulum import _make_handle, pendulum_init_params
res = {}

def counts(h):
    return np.array([h.fallback_count(), *h.fallback_causes(), h.launch_count])

def init_fields(h):
    return np.concatenate([h.fields()[k].cpu().numpy().reshape(h.n_env, -1) for k in
                           ("position_collection", "velocity_collection", "director_collection", "omega_collection")], axis=1)

def run(key, h, launches, rng, full):
    for li, k in enumerate(launches):
        a = rng.uniform(-22, 22, (h.n_env, 1)).astype(np.float32) if h.action_dim else None
        o, r, t = h.step_host(a, k)
        res[f"{key}/obs{li}"], res[f"{key}/rew{li}"], res[f"{key}/term{li}"] = o.copy(), r.copy(), t.copy()
        st = h.state_tensor().cpu().numpy()
        assert np.isfinite(st).all(), key
        res[f"{key}/state{li}"] = st if full else np.array([hashlib.blake2b(e.tobytes(), digest_size=16).digest() for e in st])
    res[f"{key}/counts"] = counts(h)

def set_fields(h, **arrays):
    fl = h.fields()
    for k, a in arrays.items():
        fl[k][:] = torch.as_tensor(a, device="cuda")
    torch.cuda.synchronize()     # (the handle steps on a stream of its own)

for n in (tl.EQ_SIZES if "eq" in cases else (512,) if "eq512" in cases else ()):
    if True:
        for size, n_env in tl.EQ_BATCHES:
            for bc in tl.LONG_BCS:
                rng = np.random.default_rng(100 * n + n_env + bc)
                h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, math=nat.MATH_FAST, **tl._eq_cfg(n, bc))
                h.reset_host(tl._random_init(rng, n_env))
                run(f"eq{n}/bc{bc}/{size}", h, tl.LAUNCHES, rng, size == "small")
                h.close()
            rng = np.random.default_rng(7 * n + n_env)
            h = _make_handle(n_env, n, tl._pendulum_dt(n), 0, nat.MATH_FAST)
            h.reset_host(pendulum_init_params(rng.random(n_env)))
            run(f"eq{n}/pendulum/{size}", h, tl.LAUNCHES, rng, size == "small")
            h.close()

if "long" in cases:
    for n in tl.LONG_SIZES:
        for bc in tl.LONG_BCS:
            h = nat.Handle(model=nat.MODEL_ROD, n_env=3, math=nat.MATH_FAST, **tl._rod_cfg(n, bc))
            h.reset_host(tl._long_init(n, bc))
            res[f"long{n}/bc{bc}/init"] = init_fields(h)
            run(f"long{n}/bc{bc}", h, tl.LAUNCHES, None, True)
            h.close()
    h = nat.Handle(model=nat.MODEL_ROD, n_env=3, math=nat.MATH_FAST, **tl._rod_cfg(2048, 1))
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
    h.close()

if "kink" in cases:
    c = tl._rod_cfg(tl.KINK_N, tl.BC_ONE_END_FIXED)
    h = nat.Handle(model=nat.MODEL_ROD, n_env=tl.KINK_ENVS, math=nat.MATH_FAST, **c)
    h.reset_host(tl._long_init(tl.KINK_N, tl.BC_ONE_END_FIXED, tl.KINK_ENVS))
    fl = h.fields()
    x, Q = (fl[k].cpu().numpy() for k in ("position_collection", "director_collection"))
    tl._kink(x, Q)
    set_fields(h, position_collection=x, director_collection=Q)
    res["kink/init"] = init_fields(h)
    run("kink", h, tl.KINK_LAUNCHES, None, True)
    h.close()

if "nan" in cases:
    for key, mk in (("rod", lambda: nat.Handle(model=nat.MODEL_ROD, n_env=4, math=nat.MATH_FAST, **tl._rod_cfg(2047, 1))),
                    ("pendulum", lambda: _make_handle(4, 2048, tl._pendulum_dt(2048), 0, nat.MATH_FAST))):
        h = mk()
        h.reset_host(pendulum_init_params(np.linspace(0.1, 0.9, 4)))
        v = h.fields()["velocity_collection"].cpu().numpy()
        v[2, 1, h.n_elem] = np.nan          # the tip node: the last thread of the last rank
        set_fields(h, velocity_collection=v)
        o, r, t = h.step_host(np.full((4, 1), 5.0, np.float32) if h.action_dim else None, 20)
        res[f"nan/{key}/term"], res[f"nan/{key}/rew"] = t.copy(), r.copy()
        h.close()

np.savez(out, **res)
"""

# SOFTROD_* settings of a worker process -> the cases it runs
SETTINGS = {"default": ({}, "eq,long,kink,nan"), "cluster": ({"SOFTROD_LEAN_CLUSTER": "1"}, "eq"),
            "safe": ({"SOFTROD_FASTPATH": "0"}, "kink"), "nofold": ({"SOFTROD_LEAN_FOLD": "0"}, "eq512")}


def _long_init(n, bc, n_env=3):
    """Three rods per handle: a random 3D orientation each (seeded by n and the BC)."""
    return _random_init(np.random.default_rng(1000 * n + bc), n_env)


def _kink(x, Q):
    """In place, on [env, ...] arrays: env KINK_DEEP and env KINK_EDGE get a KINK_DEG kink, the frames of elements
    KINK_AT[e] .. n-1 turned about their d2 and the nodes rebuilt along the turned d3."""
    n, t = KINK_N, np.deg2rad(KINK_DEG)
    for e, m in KINK_AT.items():
        ln = np.sqrt(np.sum(np.diff(x[e], axis=1) ** 2, axis=0))
        d2 = Q[e, 1, :, m]
        K = np.array([[0, -d2[2], d2[1]], [d2[2], 0, -d2[0]], [-d2[1], d2[0], 0]])
        R = np.eye(3) + np.sin(t) * K + (1 - np.cos(t)) * (K @ K)
        for k in range(m, n):
            Q[e, :, :, k] = Q[e, :, :, k] @ R.T
            x[e, :, k + 1] = x[e, :, k] + ln[k] * Q[e, 2, :, k]


@pytest.fixture(scope="module")
def worker(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("long_rods")
    script = tmp / "long_rods_worker.py"
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


def _fields(st, layout, n):
    p, v, d, w, t, k, s, dl = layout
    return {"position_collection": st[p:p + 3, :n + 1], "velocity_collection": st[v:v + 3, :n + 1],
            "director_collection": st[d:d + 9, :n].reshape(3, 3, n), "omega_collection": st[w:w + 3, :n],
            "tangents": st[t:t + 3, :n], "kappa": st[k:k + 3, :n - 1], "sigma": st[s:s + 3, :n], "dilatation": st[dl, :n]}


def _oracle(c, init_row, fields0):
    """The C oracle's rod for a GPU env, started from the x, v, Q, w the GPU held before the first launch."""
    import rod_oracle as ro
    n = c["n_elem"]
    r = ro.OracleRod(n, init_row[0:3], init_row[3:6], init_row[6:9], c["base_length"], c["base_radius"], c["density"],
                     c["youngs_modulus"], c["dt"], gravity=c["gravity"], damping_constant=c["damping_constant"],
                     bc_kind=c["bc_kind"])
    parts = np.split(fields0, np.cumsum((3 * (n + 1), 3 * (n + 1), 9 * n, 3 * n))[:-1])
    for name, a in zip(("position_collection", "velocity_collection", "director_collection", "omega_collection"), parts):
        getattr(r, name)[...] = a.reshape(getattr(r, name).shape)
    return r


def _check_vs_oracle(res, key, c, init, envs, launches, what):
    from test_parity_gpu import assert_state_close, one_ulp_divergence, rate_floors
    import rod_oracle as ro
    n, layout = c["n_elem"], res["layout"]
    mks = [functools.partial(_oracle, c, init[e], res[f"{key}/init"][e]) for e in envs]
    rods, refs = [mk() for mk in mks], [[] for _ in envs]
    for k in launches:
        ro.substeps_batch(rods, k)
        for i, o in enumerate(rods):
            refs[i].append({name: getattr(o, name).copy() for name in ORACLE_FIELDS})
    for o in rods:
        o.close()
    for i, e in enumerate(envs):
        # the oracle's one-ulp divergence over the whole horizon (measured per env, used at every launch)
        sens = one_ulp_divergence(mks[i], lambda rod: rod.substeps(sum(launches)), refs[i][-1])
        for li, ref in enumerate(refs[i]):
            f = _fields(res[f"{key}/state{li}"][e], layout, n)
            x = ref["position_collection"]
            floors = rate_floors(c["youngs_modulus"], c["density"], c["base_length"], n, c["base_radius"], np.abs(x).max())
            for name in ORACLE_FIELDS:
                assert_state_close(f[name], ref[name], name, floors, f"{what} env {e} after launch {li}", measured=sens)
            obs = res[f"{key}/obs{li}"][e]
            np.testing.assert_allclose(obs[:3], x[:, -1], rtol=2e-6, atol=1e-7)
            np.testing.assert_allclose(obs[3:6], ref["velocity_collection"][:, -1], rtol=2e-6, atol=1e-7)


# ---- 1 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", EQ_SIZES)
def test_cluster_kernel_gives_the_bits_of_the_one_cta_kernels(worker, n):
    """SOFTROD_LEAN_CLUSTER=1 (two CTAs per rod) against the default kernels (the folded-tip 512-thread kernel at
    n = 512 for plain rods, the 544 / 768 / 1024-thread CTAs otherwise): free, clamped and slider rods at random 3D
    orientations under gravity with three non-zero components, the damper on or off, and SoftPendulum-v0's model with
    random +-22 actions; 7 envs and 300 envs.  After each of two launches (400 and 600 substeps) the whole state
    block (all 32 fields; a digest per env for the 300-env batches), the observations, rewards and terminated flags
    are equal bit for bit, with no range fallback.  At n = 512 the reference is the plain model's 544-thread
    kernel (SOFTROD_LEAN_FOLD=0); the fold layout's kernel must give the same bits outside the padding slots into which
    the CTA layout writes the tip thread's pseudo-element observables (tangent, sigma and dilatation slot n, kappa
    slot n - 1), and which the folded kernel leaves alone."""
    ref, cl = worker("nofold" if n == 512 else "default"), worker("cluster")
    for model in [f"bc{bc}" for bc in LONG_BCS] + ["pendulum"]:
        for size, _ in EQ_BATCHES:
            key = f"eq{n}/{model}/{size}"
            for li in range(len(LAUNCHES)):
                for f in ("state", "obs", "rew", "term"):
                    a, b = ref[f"{key}/{f}{li}"], cl[f"{key}/{f}{li}"]
                    assert a.shape == b.shape, (key, f)
                    assert np.array_equal(a, b), (key, f, li, np.argwhere(a != b)[:5])
                if n == 512 and size == "small" and model != "pendulum":
                    fold, st = worker("default")[f"{key}/state{li}"].copy(), cl[f"{key}/state{li}"].copy()
                    for blk in (fold, st):
                        blk[:, [18, 19, 20, 24, 25, 26, 27], n] = 0.0
                        blk[:, [21, 22, 23], n - 1] = 0.0
                    assert np.array_equal(fold, st), (key, "folded", li, np.argwhere(fold != st)[:5])
            assert ref[f"{key}/counts"][0] == 0 and cl[f"{key}/counts"][0] == 0, (key, cl[f"{key}/counts"])
            assert not cl[f"{key}/term{len(LAUNCHES) - 1}"].any()


# ---- 2 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", LONG_SIZES)
def test_long_rods_vs_c_oracle(worker, n):
    """Clamped, free and slider rods of 1024-4095 elements (clusters of 3 ... 8 CTAs, the last one holding 1 ... 512
    threads), three envs each, against the C oracle started from the same state: all eight fields and the tip in the
    observation after 400 and 1000 substeps (two launches), within the 1e-9 rule of test_parity_gpu or 20x the
    oracle's own one-ulp divergence."""
    res = worker("default")
    for bc in LONG_BCS:
        c = _rod_cfg(n, bc)
        _check_vs_oracle(res, f"long{n}/bc{bc}", c, _long_init(n, bc), range(3), LAUNCHES, f"n={n} bc={bc}")
        cnt = res[f"long{n}/bc{bc}/counts"]
        assert cnt[0] == 0 and cnt[4] == 1 + 2 * len(LAUNCHES), cnt      # reset + (fast-only, fallback) per launch


@pytest.mark.gpu
def test_long_rod_handles_refuse_the_one_cta_getters(worker):
    """Rest curvature and external loads would move a long rod to kernels that cannot hold it."""
    errs = worker("default")["getter_errors"]
    assert "rest curvature is built for n_elem <= 1023" in errs[0]
    assert "external loads are built for n_elem <= 1023" in errs[1]


# ---- 3 -------------------------------------------------------------------------------------------------------------
PENDULUM_N, PENDULUM_STEPS, PENDULUM_FPS = 2048, 10, 2500   # step_skip = 1 / (2500 * 1e-6) = 400 substeps
PENDULUM_FIELDS = ("position_collection", "velocity_collection", "director_collection", "omega_collection", "tangents",
                   "dilatation")


def _pendulum_kw():
    return dict(n_elems=PENDULUM_N, time_step=_pendulum_dt(PENDULUM_N), recording_fps=PENDULUM_FPS)


class _PendulumRod:
    """An OracleSoftPendulum after reset(**reset_kw), seen as its rod (for one_ulp_divergence)."""

    def __init__(self, reset_kw):
        import rod_oracle as ro
        self.env = ro.OracleSoftPendulum(**_pendulum_kw())
        self.env.reset(**reset_kw)

    def __getattr__(self, k):
        return getattr(self.env.rod, k)

    def close(self):
        self.env.rod.close()


def _pendulum_sensitivity(reset_kw, actions):
    """The oracle's one-ulp divergence over the steps `actions` from reset(**reset_kw) (test_parity_gpu)."""
    from test_parity_gpu import one_ulp_divergence
    o = _PendulumRod(reset_kw)
    for a in actions:
        o.env.step(a)
    ref = {k: getattr(o, k).copy() for k in ORACLE_FIELDS}
    o.close()

    def advance(rod):
        for a in actions:
            rod.env.step(a)
    return one_ulp_divergence(lambda: _PendulumRod(reset_kw), advance, ref)


def _assert_pendulum_close(state, obs, rew, term, trunc, o, o_obs, o_rew, o_term, o_trunc, what, sens):
    from test_parity_gpu import assert_state_close, rate_floors
    floors = rate_floors(1e6, 1000.0, 1.0, PENDULUM_N, 0.05, np.abs(o.rod.position_collection).max())
    # the integrated state and the tangents / dilatation the outputs read; kappa and sigma of a 2048-element rod are
    # differences at round-off level (as in test_soft_pendulum_3d_golden), and test_long_rods_vs_c_oracle covers them
    for name in PENDULUM_FIELDS:
        assert_state_close(state[name], getattr(o.rod, name), name, floors, what, measured=sens)
    np.testing.assert_array_max_ulp(np.asarray(obs, np.float32), o_obs, maxulp=2)
    assert abs(float(rew) - o_rew) <= 1e-9 * max(1.0, abs(o_rew)), (what, float(rew), o_rew)
    assert (bool(term), bool(trunc)) == (o_term, o_trunc), what


@pytest.mark.gpu
def test_soft_pendulum_2048_single_env_vs_oracle():
    """gsb.make("SoftPendulum-v0", n_elems=2048) over 10 env-steps of random actions against OracleSoftPendulum."""
    import gym_softrobot_b200 as gsb
    import rod_oracle as ro
    env = gsb.make("SoftPendulum-v0", **_pendulum_kw())
    o = ro.OracleSoftPendulum(**_pendulum_kw())
    obs, _ = env.reset(seed=5)
    o_obs, _ = o.reset(seed=5)
    np.testing.assert_array_equal(obs, o_obs)
    actions = np.random.default_rng(5).uniform(-22, 22, (PENDULUM_STEPS, 1)).astype(np.float32)
    sens = _pendulum_sensitivity(dict(seed=5), actions)     # (over the whole horizon, used at every step)
    for i, a in enumerate(actions):
        obs, rew, te, tr, _ = env.step(a)
        oo, orew, ote, otr, _ = o.step(a)
        _assert_pendulum_close(env.rod_state(), obs, rew, te, tr, o, oo, orew, ote, otr, f"step {i}", sens)
    env.close()
    o.rod.close()


@pytest.mark.gpu
def test_soft_pendulum_2048_vector_env_vs_oracle():
    """gsb.make_vec("SoftPendulum-v0", 64, n_elems=2048) over 10 env-steps against the oracle (8 of the envs), with
    envs 3, 17 and 40 reset through sr_reset's env_idx after step 4 (the autoreset path): the others carry on as the
    oracle does, and the reset envs step on exactly as the envs of a fresh handle reset from the same rows (state block,
    observations, rewards and flags bit for bit)."""
    import torch
    import gym_softrobot_b200 as gsb
    import rod_oracle as ro
    from gym_softrobot_b200.envs.soft_pendulum import _make_handle, pendulum_init_params
    n_env, check, reset_ids = 64, (0, 3, 17, 31, 40, 50, 62, 63), (3, 17, 40)
    vec = gsb.make_vec("SoftPendulum-v0", n_env, autoreset=False, **_pendulum_kw())
    obs, _ = vec.reset(seed=11)
    oracles = {e: ro.OracleSoftPendulum(**_pendulum_kw()) for e in check}
    for e, o in oracles.items():
        np.testing.assert_array_equal(obs[e].cpu().numpy(), o.reset(seed=11 + e)[0])
    actions = np.random.default_rng(11).uniform(-22, 22, (PENDULUM_STEPS, n_env, 1)).astype(np.float32)
    # the oracle's one-ulp divergence over each env's whole horizon, used at every step
    sens = {e: _pendulum_sensitivity(dict(seed=11 + e), actions[:, e]) for e in check}
    init = pendulum_init_params(np.random.default_rng(99).random(len(reset_ids)))
    fresh = _make_handle(len(reset_ids), PENDULUM_N, _pendulum_dt(PENDULUM_N), 0, 0)
    fresh.reset_host(init)
    for i in range(PENDULUM_STEPS):
        if i == 5:
            idx = torch.as_tensor(reset_ids, dtype=torch.int32, device="cuda")
            vec.handle.reset(torch.as_tensor(init, device="cuda").contiguous(), idx)
        a = actions[i]
        obs, rew, te, tr, _ = vec.step(torch.as_tensor(a, device="cuda"))
        f = {k: v.cpu().numpy() for k, v in vec.fields().items()}
        for e, o in oracles.items():
            if e in reset_ids and i >= 5:
                continue
            oo, orew, ote, otr, _ = o.step(a[e])
            _assert_pendulum_close({k: f[k][e] for k in ORACLE_FIELDS}, obs[e].cpu().numpy(), rew[e], te[e], tr[e],
                                   o, oo, orew, ote, otr, f"env {e} step {i}", sens[e])
        if i >= 5:
            fo, fr, ft = fresh.step_host(np.ascontiguousarray(a[list(reset_ids)]), vec.step_skip)
            st, fst = vec.handle.state_tensor().cpu().numpy(), fresh.state_tensor().cpu().numpy()
            assert np.array_equal(st[list(reset_ids)], fst), (i, np.argwhere(st[list(reset_ids)] != fst)[:5])
            assert np.array_equal(obs[list(reset_ids)].cpu().numpy(), fo) and np.array_equal(rew[list(reset_ids)].cpu().numpy(), fr)
            assert np.array_equal(te[list(reset_ids)].cpu().numpy(), ft.astype(bool))
    fresh.close()
    vec.close()
    for o in oracles.values():
        o.rod.close()


# ---- 4 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_range_fallback_across_ctas(worker):
    """Clamped rods of n = 2047 (clusters of 4), one env kinked by 45 degrees at element 1200 (inside rank 2), one at
    elements 511 / 512 (the curvature stencil of Voronoi point 511 reads rank 1's first element).  The fast-only
    kernel flags both envs in every launch, with cause "bend" only; the state block equals the safe kernel's alone
    (SOFTROD_FASTPATH=0) bit for bit for every env after every launch, and the kinked envs match the C oracle."""
    res, safe = worker("default"), worker("safe")
    L = len(KINK_LAUNCHES)
    for li in range(L):
        for f in ("state", "obs", "rew", "term"):
            a, b = res[f"kink/{f}{li}"], safe[f"kink/{f}{li}"]
            assert np.array_equal(a, b), (f, li, np.argwhere(a != b)[:5])
    cnt = res["kink/counts"]
    assert list(cnt[:4]) == [2 * L, 0, 2 * L, 0], cnt                 # total, rotation, bend, stretch
    assert cnt[4] == 1 + 2 * L and safe["kink/counts"][4] == 1 + L, (cnt, safe["kink/counts"])
    c = _rod_cfg(KINK_N, BC_ONE_END_FIXED)
    _check_vs_oracle(res, "kink", c, _long_init(KINK_N, BC_ONE_END_FIXED, KINK_ENVS), sorted(KINK_AT), KINK_LAUNCHES,
                     "kink")


# ---- 5 -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_nan_in_the_last_rank_terminates_that_env_only(worker):
    """A NaN in the tip's velocity (the last thread of the last CTA) reaches rank 0's lead through the cluster's NaN
    flag: env 2 is terminated and no other env; SoftPendulum-v0's reward for it is -50."""
    res = worker("default")
    for key in ("rod", "pendulum"):
        assert list(res[f"nan/{key}/term"]) == [0, 0, 1, 0], (key, res[f"nan/{key}/term"])
    rew = res["nan/pendulum/rew"]
    assert rew[2] == -50.0 and np.isfinite(rew).all() and (rew[[0, 1, 3]] >= 0).all(), rew
