"""GPU parity: CUDA path (through the C-ABI) vs golden fixtures and the C oracle.

Tolerances (BASELINE.json north_star): FP64 state to rel 1e-9 over 1000 substeps,
where "rel" is max|a-b| / max|b| per field; termination/truncation bit-exact;
observations are float32 casts of FP64 values (compared to 2 float32 ulp); rewards
are FP64 functions of the state (compared to 1e-9 — they cannot be bit-exact
unless the state is, see DESIGN.md).
"""
import os
import time

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOL = 1e-9
FIELDS = {"position": "position_collection", "velocity": "velocity_collection",
          "director": "director_collection", "omega": "omega_collection",
          "tangents": "tangents", "kappa": "kappa", "sigma": "sigma", "dilatation": "dilatation"}


def rel(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def _native():
    from gym_softrobot_b200 import _native as nat
    return nat


def rate_floors(E, rho, L, n, r, max_abs_x):
    """Round-off floor of a configuration: absolute coordinates of size |x| resolve an element's strain only to
    eps |x| / dl per substep in ANY implementation (the oracle included); through the axial stiffness that is a
    velocity noise of ~ eps |x| c / dl (c = sqrt(E/rho)) and ~ that / r for omega.  A rod that has barely
    started to move must be compared against this floor as well as against the relative tolerance."""
    fv = 64 * 2.2e-16 * max(max_abs_x, L) * np.sqrt(E / rho) / (L / n)
    return {"position_collection": 0.0, "director_collection": 0.0, "velocity_collection": fv,
            "omega_collection": fv / r}


# a rate field counts as "the rod has barely started to move" below these magnitudes; only then may the absolute
# round-off floor of rate_floors() stand in for the relative bound
TINY_RATE = {"velocity_collection": 1e-2, "omega_collection": 1e-1}
# Magnitude floors of the strain fields: a straight rod at rest holds kappa / sigma of pure round-off size (computed by
# cancellation: axial(Q+ Q^T) / D, e Q t - z), where "relative to max|ref|" is meaningless; they are compared relative
# to max(|ref|, the magnitude a gently loaded rod reaches): 1e-3 1/m of curvature, 1e-6 of strain.
STRAIN_FLOOR = {"kappa": 1e-3, "sigma": 1e-6}


def assert_state_close(mine, ref, name, floors, what, tol=TOL, measured=None):
    """max|mine - ref| <= tol * max|ref|.  Two documented ways out, nothing else:
    * `measured` (name -> abs divergence of the ORACLE from itself when its input positions move by one ulp, see
      one_ulp_divergence): up to 20x that — the reference cannot reproduce its own numbers better than this;
    * a rate field whose reference magnitude is still tiny (TINY_RATE) may meet the absolute round-off floor of
      rate_floors() instead."""
    scale, err = float(np.abs(ref).max()), float(np.abs(mine - ref).max())
    if err <= tol * max(scale, STRAIN_FLOOR.get(name, 0.0)):
        return
    if measured is not None and err <= 20.0 * measured.get(name, 0.0):
        return
    ok = name in TINY_RATE and scale < TINY_RATE[name] and err <= tol * scale + floors.get(name, 0.0)
    assert ok, (f"{what} {name}: abs err {err:.3e}, rel {err / max(scale, 1e-300):.3e} (|ref| {scale:.3e}, floor "
                f"{floors.get(name, 0.0):.2e}, one-ulp divergence of the oracle {(measured or {}).get(name, 0.0):.2e})")


def one_ulp_divergence(make_rod, advance, ref, n_rep=2):
    """How far the C oracle moves from its own result `ref` (name -> array) when every initial position coordinate is
    nudged to a neighbouring double: the round-off sensitivity of the configuration, measured instead of estimated.
    (Thin, finely discretised rods amplify position round-off through eps |x| / dl strains: 3e-9 rad/s on
    |w| = 0.6 rad/s for n_elem = 1023, r = 4 mm after 1000 substeps.)"""
    out = {k: 0.0 for k in ref}
    for rep in range(n_rep):
        rng = np.random.default_rng(4242 + rep)
        rod = make_rod()
        x = rod.position_collection
        x[...] = np.nextafter(x, np.where(rng.random(x.shape) < 0.5, -np.inf, np.inf))
        advance(rod)
        for k in ref:
            out[k] = max(out[k], float(np.abs(getattr(rod, k) - ref[k]).max()))
        rod.close()
    return out


def fma_build_divergence(make_rod, advance, ref):
    """The second measured conditioning floor: how far the SAME C source built with FMA contraction (oracle/Makefile,
    rod_oracle.variant("fma")) ends from the default build.  Unlike the one-ulp start above, the two builds round
    differently in every substep — which is also how a CUDA kernel differs from either."""
    import rod_oracle as ro
    with ro.variant("fma"):
        rod = make_rod()
    advance(rod)
    out = {k: float(np.abs(getattr(rod, k) - ref[k]).max()) for k in ref}
    rod.close()
    return out


# ---- multi-rod assemblies against the multi-rod C oracle (VERDICT r1 item 1) ------------------------------------
# Scale floors of the assembly comparisons: a field is compared relative to max|ref| over the arm, but not below
# the magnitude it has once the arm is actuated (a straight arm at rest holds kappa / sigma / rates of pure
# round-off size, where "relative" is meaningless).  Same table as tests/test_oracle_golden.py.
ASM_FLOOR = dict(position_collection=1e-2, velocity_collection=1e-3, director_collection=1.0, omega_collection=1e-2,
                 tangents=1.0, kappa=1.0, sigma=1e-3, dilatation=1.0)


def _asm_err(mine, ref, key):
    return float(np.abs(mine - ref).max() / max(np.abs(ref).max(), ASM_FLOOR[key]))


def make_pendulum_handle(n_env, math, n_elem=50, dt=1e-4):
    from gym_softrobot_b200.envs.soft_pendulum import _make_handle
    return _make_handle(n_env, n_elem, dt, 0, math)


def u01_for_seed(seed):
    return np.random.Generator(np.random.PCG64(np.random.SeedSequence(seed))).random()


@pytest.mark.parametrize("math", [0, 1], ids=["fast", "faithful"])
def test_golden_substeps(golden_dir, math):
    """State after 1/10/100/400/1000 raw substeps vs the reference-env-on-shim fixture."""
    import torch
    from gym_softrobot_b200.envs.soft_pendulum import pendulum_init_params
    g = np.load(os.path.join(golden_dir, "soft_pendulum_seed42_substeps.npz"))
    h = make_pendulum_handle(1, math)
    h.reset_host(pendulum_init_params(u01_for_seed(42)))
    act = np.array([[g["action"]]], dtype=np.float32)
    done = 0
    for target in (1, 10, 100, 400, 1000):
        h.step_host(act, target - done)
        done = target
        torch.cuda.synchronize()
        f = {k: v[0].cpu().numpy() for k, v in h.fields().items()}
        # (after 1 and 10 substeps the rod has not started to move: |w| ~ 1e-13 rad/s of pure round-off)
        floors = rate_floors(1e6, 1000.0, 1.0, 50, 0.05, 1.0)
        for gk, fk in FIELDS.items():
            assert_state_close(f[fk], g[f"sub{target}/{gk}"], fk, floors, f"math={math} substeps={target}")
    h.close()


@pytest.mark.parametrize("math", [0, 1], ids=["fast", "faithful"])
def test_golden_episode_single_env(golden_dir, math):
    """Config 1 of BASELINE.json: seed 42, the recorded random actions, through the Gymnasium façade."""
    import gym_softrobot_b200 as gsb
    g = np.load(os.path.join(golden_dir, "soft_pendulum_seed42_episode.npz"))
    env = gsb.make("SoftPendulum-v0", math=math)
    obs0, info = env.reset(seed=42)
    assert obs0.dtype == np.float32 and np.array_equal(obs0, g["obs0"])
    n_check = 30  # 12000 substeps; the full 126-step episode is checked for flags/time only below
    for i in range(n_check):
        obs, r, te, tr, info = env.step(g["actions"][i])
        assert te == bool(g["terminated"][i]) and tr == bool(g["truncated"][i])
        assert info["time"] == g["time"][i]  # float64 time accumulation is bit-exact
        assert isinstance(te, bool) and isinstance(tr, bool) and np.isscalar(r)
        if i < 3:  # 1200 substeps: the 1e-9 window of the north star
            st = env.rod_state()
            for gk, fk in FIELDS.items():
                assert_state_close(st[fk], g[f"state{i + 1}/{gk}"], fk, {}, f"step {i}")
            assert abs(r - g["reward"][i]) <= TOL * max(1.0, abs(g["reward"][i]))
        np.testing.assert_allclose(obs, g["obs"][i], rtol=2e-6, atol=1e-7)
        assert abs(r - g["reward"][i]) <= 1e-6 * max(1.0, abs(g["reward"][i]))
    env.close()


def test_golden_episode_flags_full(golden_dir):
    """Whole 126-step episode: termination/truncation sequence and info['time'] bit-exact."""
    import gym_softrobot_b200 as gsb
    g = np.load(os.path.join(golden_dir, "soft_pendulum_seed42_episode.npz"))
    env = gsb.make("SoftPendulum-v0")
    env.reset(seed=42)
    n = int(g["n_steps"])
    for i in range(n):
        obs, r, te, tr, info = env.step(g["actions"][i])
        assert (te, tr) == (bool(g["terminated"][i]), bool(g["truncated"][i])), i
        assert info["time"] == g["time"][i]
    assert tr and not te
    # long-horizon drift stays small even after 50400 substeps
    np.testing.assert_allclose(obs, g["obs"][n - 1], rtol=1e-4, atol=1e-5)
    env.close()


def test_reference_determinism_protocol(golden_dir):
    """The reference's own test (tests/envs/test_determinism.py:7-58): two envs, seed 0, 3 steps, exact equality."""
    import gym_softrobot_b200 as gsb
    g = np.load(os.path.join(golden_dir, "softpendulum_v0_determinism_seed0.npz"))
    runs = []
    for _ in range(2):
        env = gsb.make("SoftPendulum-v0")
        o0, _ = env.reset(seed=0)
        env.action_space.seed(0)
        acts = [env.action_space.sample() for _ in range(3)]
        resp = [env.step(a) for a in acts]
        env.close()
        runs.append((o0, acts, resp))
    (o1, a1, r1), (o2, a2, r2) = runs
    assert np.array_equal(o1, o2) and np.array_equal(o1, g["obs0"])
    for x, y, ga in zip(a1, a2, g["actions"]):
        assert np.array_equal(x, y) and np.array_equal(x, ga)
    for (ob1, rw1, t1, x1, _), (ob2, rw2, t2, x2, _), gob, grw in zip(r1, r2, g["obs"], g["reward"]):
        np.testing.assert_array_equal(ob1, ob2)
        assert rw1 == rw2 and t1 == t2 and x1 == x2
        np.testing.assert_allclose(ob1, gob, rtol=2e-6, atol=1e-7)
        assert abs(rw1 - grw) < 1e-9


@pytest.mark.parametrize("n_env", [1, 5, 128, 4096])
def test_batched_vs_oracle(n_env):
    """Batched kernel vs the C oracle on seeded per-env initial angles and actions (1200 substeps)."""
    import torch
    import rod_oracle
    import gym_softrobot_b200 as gsb
    env = gsb.make_vec("SoftPendulum-v0", n_env, autoreset=False)
    obs, _ = env.reset(seed=42)
    check = sorted(set([0, n_env - 1] + list(np.random.default_rng(1).integers(0, n_env, size=6))))
    oracles = {i: rod_oracle.OracleSoftPendulum() for i in check}
    for i, o in oracles.items():
        o_obs, _ = o.reset(seed=42 + i)
        assert np.array_equal(obs[i].cpu().numpy(), o_obs)
    gen = torch.Generator(device="cuda").manual_seed(42)
    for step in range(3):
        a = (torch.rand((n_env, 1), generator=gen, device="cuda") * 44 - 22).float()
        obs, rew, term, trunc, info = env.step(a)
        f = {k: v.cpu().numpy() for k, v in env.fields().items()}
        a_np = a.cpu().numpy()
        for i, o in oracles.items():
            ob, r, te, tr, oi = o.step(a_np[i])
            for name in ("position_collection", "velocity_collection", "director_collection",
                         "omega_collection", "tangents"):
                err = rel(f[name][i], getattr(o.rod, name))
                assert err < TOL, f"n_env={n_env} env={i} step={step} {name}: {err:.3e}"
            assert bool(term[i]) == te and bool(trunc[i]) == tr
            assert abs(float(rew[i]) - r) <= TOL * max(1.0, abs(r))
            np.testing.assert_allclose(obs[i].cpu().numpy(), ob, rtol=2e-6, atol=1e-7)
            assert float(info["time"][i]) == oi["time"]
    env.close()


def test_full_size_properties():
    """BASELINE config 2 (4096 envs, n=50): size-independent properties.

    (a) run-to-run determinism is bit-exact; (b) envs with identical seeds and actions
    produce bit-identical states wherever they sit in the batch; (c) state stays finite.
    """
    import torch
    from gym_softrobot_b200.envs.soft_pendulum import pendulum_init_params
    n_env = 4096
    u = np.random.default_rng(7).random(64)
    u_all = np.tile(u, n_env // 64)
    act = torch.as_tensor(np.tile(np.random.default_rng(8).uniform(-22, 22, 64), n_env // 64)
                          .astype(np.float32).reshape(n_env, 1), device="cuda")
    outs = []
    for _ in range(2):
        h = make_pendulum_handle(n_env, 0)
        h.reset(torch.as_tensor(pendulum_init_params(u_all), device="cuda").contiguous())
        obs = torch.empty((n_env, 4), dtype=torch.float32, device="cuda")
        rew = torch.empty(n_env, dtype=torch.float64, device="cuda")
        term = torch.empty(n_env, dtype=torch.uint8, device="cuda")
        for _s in range(2):
            h.step(act, 400, obs, rew, term)
        torch.cuda.synchronize()
        outs.append((h.state_tensor().clone(), obs.clone(), rew.clone(), term.clone()))
        h.close()
    (s1, o1, r1, t1), (s2, o2, r2, t2) = outs
    assert torch.equal(s1, s2) and torch.equal(o1, o2) and torch.equal(r1, r2)
    assert int(t1.sum()) == 0 and bool(torch.isfinite(s1).all())
    s = s1.reshape(n_env // 64, 64, *s1.shape[1:])
    assert torch.equal(s[0].expand_as(s), s), "identical envs diverged across the batch"


def test_free_fall_and_nan_guard():
    """PositionVerlet is exact for constant acceleration (free rod, no damping); NaN -> terminated."""
    import torch
    nat = _native()
    h = nat.Handle(model=nat.MODEL_ROD, n_env=3, n_elem=20, dt=1e-4, base_length=1.0, base_radius=0.05,
                   density=1000.0, youngs_modulus=1e6, gravity=(0.0, -9.80665, 0.0))
    init = np.zeros((3, 9)); init[:, 3] = 1.0; init[:, 7] = 1.0
    h.reset_host(init)
    y0 = h.fields()["position_collection"][:, 1].clone()
    obs, rew, term = h.step_host(None, 1000)
    t = 0.1
    y = h.fields()["position_collection"][:, 1]
    assert float((y - y0 - 0.5 * -9.80665 * t * t).abs().max()) < 1e-13
    assert term.sum() == 0
    h.fields()["velocity_collection"][1, 0, 3] = float("nan")
    obs, rew, term = h.step_host(None, 2)
    assert list(term) == [0, 1, 0]
    h.close()


def _tilted_init(n_env, seed=42, max_deg=5.0):
    """Config 3 of BASELINE.json: horizontal rod, per-env tilt of +-5 degrees about z (seeded)."""
    ang = np.deg2rad(np.array([np.random.Generator(np.random.PCG64(np.random.SeedSequence(seed + i))).uniform(
        -max_deg, max_deg) for i in range(n_env)]))
    init = np.zeros((n_env, 9))
    init[:, 3], init[:, 4] = np.cos(ang), np.sin(ang)      # direction
    init[:, 6], init[:, 7] = -np.sin(ang), np.cos(ang)     # normal (perpendicular, in plane)
    return init


@pytest.mark.parametrize("n_elem,dt,radius", [(100, 5e-5, 0.025), (20, 1e-4, 0.05), (63, 5e-5, 0.03), (200, 2e-5, 0.025),
                                              (3, 1e-4, 0.05), (4, 1e-4, 0.05), (255, 1e-5, 0.01), (1023, 2e-6, 0.004),
                                              (512, 5e-6, 0.008)])     # 512: the lean kernel's fold layout
def test_generic_rod_vs_oracle(n_elem, dt, radius):
    """BASELINE config 3 family: clamped rod (OneEndFixedBC) + gravity + analytical damping, no action."""
    import rod_oracle as ro
    nat = _native()
    n_env = 7
    init = _tilted_init(n_env)
    h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n_elem, dt=dt, base_length=1.0, base_radius=radius,
                   density=1000.0, youngs_modulus=1e6, gravity=(0.0, -9.80665, 0.0), damping_constant=2e-3,
                   bc_kind=nat.BC_ONE_END_FIXED)
    h.reset_host(init)
    rods = [ro.OracleRod(n_elem, init[i, 0:3], init[i, 3:6], init[i, 6:9], 1.0, radius, 1000.0, 1e6, dt,
                         gravity=(0.0, -9.80665, 0.0), damping_constant=2e-3, bc_kind=ro.BC_ONE_END_FIXED)
            for i in range(n_env)]
    names = ("position_collection", "velocity_collection", "director_collection", "omega_collection")
    done = 0
    for chunk in (400, 600):   # 1000 substeps in two launches
        obs, rew, term = h.step_host(None, chunk)
        done += chunk
        f = {k: v.cpu().numpy() for k, v in h.fields().items()}
        for i, r in enumerate(rods):
            r.substeps(chunk)
            floors = rate_floors(1e6, 1000.0, 1.0, n_elem, radius, np.abs(r.position_collection).max())
            measured = None
            if i == 0:    # the oracle's own one-ulp sensitivity for this configuration (same for every env)
                mk = lambda: ro.OracleRod(n_elem, init[0, 0:3], init[0, 3:6], init[0, 6:9], 1.0, radius, 1000.0, 1e6, dt,
                                          gravity=(0.0, -9.80665, 0.0), damping_constant=2e-3, bc_kind=ro.BC_ONE_END_FIXED)
                sens = one_ulp_divergence(mk, lambda rod: rod.substeps(done), {k: getattr(r, k).copy() for k in names})
            for name in names:
                assert_state_close(f[name][i], getattr(r, name), name, floors, f"n={n_elem} env={i}", measured=sens)
            np.testing.assert_allclose(obs[i, :3], r.position_collection[:, -1], rtol=2e-6, atol=1e-7)
        assert term.sum() == 0
    h.close()


def test_soft_pendulum_3d_golden(golden_dir):
    """§8 f1: SoftPendulum3D-v0 through the Gymnasium facade vs the reference-env-on-shim fixture."""
    import gym_softrobot_b200 as gsb
    g = np.load(os.path.join(golden_dir, "soft_pendulum_3d_seed42.npz"))
    env = gsb.make("SoftPendulum3D-v0")
    obs0, _ = env.reset(seed=42)
    assert obs0.dtype == np.float32 and obs0.shape == (9,)
    np.testing.assert_array_equal(obs0, g["obs0"])
    for i, a in enumerate(g["actions"]):
        obs, r, te, tr, info = env.step(a)
        st = env.rod_state()
        for gk, fk in FIELDS.items():
            if gk in ("kappa", "sigma"):
                continue
            err = rel(st[fk], g[f"state{i + 1}/{gk}"])
            assert err < TOL, f"step {i} field {gk} rel err {err:.3e}"
        np.testing.assert_allclose(obs, g["obs"][i], rtol=2e-6, atol=1e-7)
        assert abs(r - g["reward"][i]) < 1e-9 and abs(info["tilt"] - g["tilt"][i]) < 1e-9
        assert (te, tr) == (bool(g["terminated"][i]), bool(g["truncated"][i]))
        assert isinstance(r, float) and isinstance(te, bool) and isinstance(tr, bool)
    with pytest.raises(ValueError):
        env.step(np.array([2.0, 0.0], dtype=np.float32))
    env.close()


def test_soft_pendulum_3d_batched_vs_oracle():
    import torch
    import rod_oracle
    import gym_softrobot_b200 as gsb
    n_env = 300
    env = gsb.make_vec("SoftPendulum3D-v0", n_env, autoreset=False)
    obs, _ = env.reset(seed=7)
    check = [0, 1, 150, 299]
    oracles = {i: rod_oracle.OracleSoftPendulum3D() for i in check}
    for i, o in oracles.items():
        o_obs, _ = o.reset(seed=7 + i)
        np.testing.assert_array_equal(obs[i].cpu().numpy(), o_obs)
    gen = torch.Generator(device="cuda").manual_seed(3)
    for step in range(3):
        a = (torch.rand((n_env, 2), generator=gen, device="cuda") * 2 - 1).float()
        obs, rew, term, trunc, info = env.step(a)
        f = {k: v.cpu().numpy() for k, v in env.fields().items()}
        a_np = a.cpu().numpy()
        for i, o in oracles.items():
            ob, r, te, tr, oi = o.step(a_np[i])
            for name in ("position_collection", "velocity_collection", "director_collection", "omega_collection"):
                err = rel(f[name][i], getattr(o.rod, name))
                assert err < TOL, f"env={i} step={step} {name}: {err:.3e}"
            np.testing.assert_allclose(obs[i].cpu().numpy(), ob, rtol=2e-6, atol=1e-7)
            assert abs(float(rew[i]) - r) < 1e-9 and bool(term[i]) == te and bool(trunc[i]) == tr
            assert abs(float(info["tilt"][i]) - oi["tilt"]) < 1e-9
    env.close()


def test_fp32_mode_accuracy():
    """Optional FP32 mode (north star: 1e-4 over 1000 substeps), all four integrated fields after 1200 substeps.
    SR_DTYPE_F32 stores the state in FP32 and evaluates stresses, couples and the damper in FP32; the kinematic update,
    the edge vectors, Q dx and Q+ Q^T stay FP64 inside a launch (rod_kernel_lean.cuh) — an all-FP32 step is limited by
    the strain's cancellation, not by accumulation (round 1: velocities 4e-4, omega 2e-3).  omega is compared on the
    elements the reference integrates sensibly; the base element's w1, which the reference env lets run away to ~1e5
    rad/s (DESIGN.md §4.1), is compared relative to itself."""
    import rod_oracle
    from gym_softrobot_b200.envs.soft_pendulum import pendulum_init_params
    nat = _native()
    n_env = 4
    u = np.random.default_rng(0).random(n_env)
    acts = np.random.default_rng(1).uniform(-22, 22, size=(3, n_env, 1)).astype(np.float32)
    from gym_softrobot_b200.envs.soft_pendulum import _make_handle
    h = _make_handle(n_env, 50, 1e-4, 0, nat.MATH_FAST, nat.DTYPE_F32)
    h.reset_host(pendulum_init_params(u))
    orc = [rod_oracle.OracleSoftPendulum() for _ in range(n_env)]
    for i, o in enumerate(orc):
        o.reset(u01=u[i])
    worst = {}
    for s in range(3):   # 1200 substeps
        obs, rew, term = h.step_host(acts[s], 400)
        f = {k: v.double().cpu().numpy() for k, v in h.fields().items()}
        for i, o in enumerate(orc):
            ob, r, te, tr, _ = o.step(acts[s][i])
            errs = {"position": rel(f["position_collection"][i], o.rod.position_collection),
                    "director": rel(f["director_collection"][i], o.rod.director_collection),
                    "velocity": rel(f["velocity_collection"][i], o.rod.velocity_collection),
                    "omega": rel(f["omega_collection"][i][:, 1:], o.rod.omega_collection[:, 1:]),
                    "omega_base": rel(f["omega_collection"][i][:, 0], o.rod.omega_collection[:, 0])}
            for k, e in errs.items():
                worst[k] = max(worst.get(k, 0.0), e)
                assert e < 1e-4, f"step {s} env {i} {k}: {e:.3e}"
            np.testing.assert_allclose(obs[i], ob, rtol=1e-4, atol=1e-4)
            assert bool(term[i]) == te
    print("fp32 mode after 1200 substeps:", {k: f"{e:.1e}" for k, e in worst.items()})
    assert h.state_tensor().dtype.itemsize == 4
    h.close()


def _arm_contact(before_forcing=True):
    from gym_softrobot_b200.envs.arm_single import arm_contact_params
    return arm_contact_params(before_forcing=before_forcing)


@pytest.mark.parametrize("before_forcing", [True, False], ids=["contact-first", "forcing-first"])
def test_plane_contact_friction_vs_oracle(before_forcing):
    """§8 a14 + a16: free rod on a frictional plane, per-env rest curvature, both synchronize orders (B-1)."""
    import torch
    import rod_oracle as ro
    from gym_softrobot_b200.envs.arm_single import curvature_interp_matrix, _ROD
    nat = _native()
    n_env, n, dt = 6, 50, 7e-5
    c = _arm_contact(before_forcing)
    h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n, dt=dt, gravity=(0.0, 0.0, -9.81), damping_constant=1e-2,
                   bc_kind=nat.BC_FREE, contact=c, **_ROD)
    init = np.zeros((n_env, 9)); init[:, 3] = 1.0; init[:, 8] = 1.0
    h.reset_host(init)
    W = curvature_interp_matrix(7, n - 1)
    rng = np.random.default_rng(5)
    rods = [ro.OracleRod(n, [0, 0, 0], [1.0, 0, 0], [0, 0, 1.0], _ROD["base_length"], _ROD["base_radius"], 1000.0, 1e6, dt,
                         gravity=(0.0, 0.0, -9.81), damping_constant=1e-2, contact=c) for _ in range(n_env)]
    for step in range(3):
        acts = rng.uniform(-10, 10, size=(n_env, 7))
        rk = acts @ W.T
        h.rest_kappa_tensor()[:, 0, :] = torch.as_tensor(rk, device="cuda")
        obs, rew, term = h.step_host(None, 400)
        f = {k: v.cpu().numpy() for k, v in h.fields().items()}
        for i, r in enumerate(rods):
            r.rest_kappa[0, :] = rk[i]
            r.substeps(400)
            for name in ("position_collection", "velocity_collection", "director_collection", "omega_collection"):
                err = rel(f[name][i], getattr(r, name))
                assert err < TOL, f"step={step} env={i} {name}: {err:.3e}"
    # the rod must actually be resting on the plane (contact active), not falling through or floating
    z = f["position_collection"][:, 2, :]
    assert z.min() > -1e-3 and z.max() < 0.05
    h.close()


def test_arm_single_env_golden(golden_dir):
    """OctoArmSingle-v0 through the Gymnasium facade vs the reference-env-on-shim fixture."""
    import gym_softrobot_b200 as gsb
    g = np.load(os.path.join(golden_dir, "octo_arm_single_seed42.npz"))
    env = gsb.make("OctoArmSingle-v0")
    obs0, _ = env.reset(seed=42)
    assert obs0.dtype == np.float32 and obs0.shape == (25,)
    np.testing.assert_allclose(obs0, g["obs0"], rtol=1e-6, atol=1e-6)
    for i, a in enumerate(g["actions"]):
        obs, r, te, tr, info = env.step(a)
        st = env.rod_state()
        # 714 substeps per env-step: the first step is inside the north star's 1000-substep window (1e-9, every field);
        # the later ones (up to 3570 substeps) get 1e-8
        for gk, fk in FIELDS.items():
            assert_state_close(st[fk], g[f"state{i + 1}/{gk}"], fk, {}, f"step {i}", tol=TOL if i == 0 else 1e-8)
        np.testing.assert_allclose(obs, g["obs"][i], rtol=1e-4, atol=1e-5)
        assert abs(r - float(g["reward"][i])) < 1e-6
        assert (te, tr) == (bool(g["terminated"][i]), bool(g["truncated"][i]))
    env.close()


def test_octo_flat_env_golden(golden_dir):
    """§8 a12/a13/a15 (config 4 topology): OctoFlat-v0 — 8 arms + rigid head + FixedJoint2Rigid joints +
    plane contact — through the Gymnasium facade vs the reference-env-on-shim fixture (recording_fps=50)."""
    import gym_softrobot_b200 as gsb
    g = np.load(os.path.join(golden_dir, "octo_flat_seed42.npz"))
    env = gsb.make("OctoFlat-v0", recording_fps=int(g["recording_fps"]))
    assert env.step_skip == int(g["step_skip"])
    obs0, _ = env.reset(seed=42)
    np.testing.assert_allclose(env._target, g["target"], rtol=0, atol=0)
    np.testing.assert_allclose(obs0["individual"], g["obs0/individual"], rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(obs0["shared"], g["obs0/shared"], rtol=1e-6, atol=1e-7)
    for i, a in enumerate(g["actions"]):
        obs, r, te, tr, info = env.step(a)
        st = env.state()
        # 3 x 285 = 855 substeps in total: inside the 1000-substep window, 1e-9 on every field (kappa, sigma included)
        for arm in range(8):
            for gk, fk in FIELDS.items():
                err = _asm_err(st[fk][arm], g[f"state{i + 1}/arm{arm}/{gk}"], fk)
                assert err < TOL, f"step {i} arm {arm} {gk}: {err:.3e}"
        hd = st["head"]
        for sl, gk, fk in ((slice(0, 3), "position", "position_collection"), (slice(3, 6), "velocity", "velocity_collection"),
                           (slice(6, 15), "director", "director_collection"), (slice(15, 18), "omega", "omega_collection")):
            err = _asm_err(hd[sl], g[f"state{i + 1}/head/{gk}"].reshape(-1), fk)
            assert err < TOL, f"step {i} head {gk}: {err:.3e}"
        np.testing.assert_allclose(obs["individual"], g[f"obs{i + 1}/individual"], rtol=1e-4, atol=1e-5)
        np.testing.assert_allclose(obs["shared"], g[f"obs{i + 1}/shared"], rtol=1e-4, atol=1e-6)
        assert abs(r - float(g["reward"][i])) < 1e-6
        assert (te, tr) == (bool(g["terminated"][i]), bool(g["truncated"][i]))
    env.close()


def test_octo_flat_batched_consistency():
    """Batched OctoFlat: envs are independent — every env fed the same actions evolves bit-identically
    wherever it sits in the batch / CTA, and matches a batch of one."""
    import torch
    import gym_softrobot_b200 as gsb
    acts = torch.as_tensor(np.random.default_rng(3).uniform(-22, 22, size=(2, 24)).astype(np.float32), device="cuda")
    outs = []
    for n_env in (1, 37):
        env = gsb.make_vec("OctoFlat-v0", n_env, recording_fps=100, autoreset=False)
        env.reset(seed=5)
        for s in range(2):
            obs, rew, term, trunc, info = env.step(acts[s].expand(n_env, 24))
        torch.cuda.synchronize()
        outs.append((env.handle.state_tensor().clone(), env.handle.head_tensor().clone(), rew.clone()))
        assert int(term.sum()) == 0
        env.close()
    (s1, h1, r1), (s37, h37, r37) = outs
    s37 = s37.reshape(37, 8, *s37.shape[1:])
    assert torch.equal(s37[0].expand_as(s37), s37) and torch.equal(h37[0].expand_as(h37), h37)
    assert torch.equal(s37[0], s1.reshape(8, *s1.shape[1:])) and torch.equal(h37[0], h1[0])
    assert torch.isfinite(s37).all()


@pytest.mark.parametrize("before_forcing", [True, False], ids=["contact-first", "forcing-first"])
def test_long_slender_rod_with_contact_fp64_and_fp32(before_forcing):
    """BASELINE config 5: long slender rod, n_elem = 512, ground contact + anisotropic friction,
    FP64 vs oracle and the FP32 mode next to it (positions / directors to 1e-4).

    contact-first: the plane sees no weight, so friction is off and the comparison is round-off
    limited (1e-9).  forcing-first (the envs' order): the rod starts at rest and its elements pass
    slowly through the regularised stick-slip band |v| in [tol, 2 tol] = [1e-8, 2e-8] m/s, where the
    reference's slip function has slope 1/tol: one explicit substep multiplies a velocity difference
    by dt mu g / tol ~ 4e2, so two correct implementations chatter apart up to the friction-force
    scale (measured 9e-10 m, 4e-7 in the directors (roll), 6e-4 of |v|max after 400 substeps); the bounds
    below are that scale."""
    import torch
    import rod_oracle as ro
    from gym_softrobot_b200.envs.arm_single import arm_contact_params
    nat = _native()
    n, dt, L, r = 512, 5e-6, 1.0, 0.005
    c = arm_contact_params(before_forcing=before_forcing)
    c["plane_origin"] = [0.0, 0.0, -r]
    rod_kw = dict(base_length=L, base_radius=r, density=1000.0, youngs_modulus=1e6)
    n_env = 3
    init = np.zeros((n_env, 9)); init[:, 3] = 1.0; init[:, 8] = 1.0
    rk = np.random.default_rng(9).uniform(-3, 3, size=(n_env, 1)) * np.sin(np.linspace(0, 3 * np.pi, n - 1))[None, :]
    rods = [ro.OracleRod(n, [0, 0, 0], [1.0, 0, 0], [0, 0, 1.0], L, r, 1000.0, 1e6, dt, gravity=(0.0, 0.0, -9.81),
                         damping_constant=1e-2, contact=c) for _ in range(n_env)]
    for i, o in enumerate(rods):
        o.rest_kappa[0, :] = rk[i]
        o.substeps(400)
    # rates (contact-first): the rod has barely started to move after 2 ms (|v|max ~ 1.5e-4 m/s) while position
    # round-off (1e-16 m) times the stiff frequency c/dl = 1.6e4 1/s is ~2e-12 m/s: the relative floor is ~1e-8
    tol64 = (TOL, TOL, 1e-7) if before_forcing else (1e-8, 5e-6, 5e-3)
    for dtype, tol_x, tol_q, tol_r in ((nat.DTYPE_F64, *tol64), (nat.DTYPE_F32, 1e-4, 1e-4, None)):
        h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n, dt=dt, gravity=(0.0, 0.0, -9.81),
                       damping_constant=1e-2, bc_kind=nat.BC_FREE, contact=c, dtype=dtype, **rod_kw)
        h.reset_host(init)
        h.rest_kappa_tensor()[:, 0, :] = torch.as_tensor(rk, device="cuda").to(h.rest_kappa_tensor().dtype)
        obs, rew, term = h.step_host(None, 400)
        f = {k: v.double().cpu().numpy() for k, v in h.fields().items()}
        assert term.sum() == 0
        for i, o in enumerate(rods):
            assert rel(f["position_collection"][i], o.position_collection) < tol_x
            assert rel(f["director_collection"][i], o.director_collection) < tol_q
            if tol_r is not None:
                assert rel(f["velocity_collection"][i], o.velocity_collection) < tol_r
                # roll rate: chatter amplitude dt mu g / r on top of |w| ~ 0.7 rad/s (measured 9e-3)
                assert rel(f["omega_collection"][i], o.omega_collection) < (tol_r if before_forcing else 3e-2)
        h.close()


def _random_rod_case(rng):
    n = int(rng.integers(5, 121))
    L = float(rng.uniform(0.3, 2.0))
    r = float(L / n * rng.uniform(0.4, 1.6))          # element aspect ratio around 1
    E = float(10 ** rng.uniform(5.0, 7.0))
    rho = float(rng.uniform(500, 4000))
    dl = L / n
    dt = float(0.005 * dl / np.sqrt(E / rho) * rng.uniform(0.5, 1.5)) * 10   # ~5 % of the axial CFL limit
    g = rng.normal(size=3); g = 9.81 * g / np.linalg.norm(g)
    damping = float(10 ** rng.uniform(-3, 0)) if rng.random() < 0.8 else -1.0
    bc = int(rng.choice([0, 1]))                          # free / one end fixed
    d = rng.normal(size=3); d /= np.linalg.norm(d)
    nn = np.cross(d, rng.normal(size=3)); nn /= np.linalg.norm(nn)
    start = rng.uniform(-1, 1, size=3)
    return dict(n=n, L=L, r=r, E=E, rho=rho, dt=dt, g=g, damping=damping, bc=bc, init=np.concatenate([start, d, nn]))


@pytest.mark.parametrize("seed", range(12))
def test_randomized_rods_vs_oracle(seed):
    """Seeded random rods (n_elem 5..120, arbitrary orientation, material, gravity direction, damping, BC)
    through both kernels vs the C oracle: 300 substeps, state to 1e-9 (rates: plus the configuration's
    own round-off floor, see below)."""
    import rod_oracle as ro
    nat = _native()
    c = _random_rod_case(np.random.default_rng(1000 + seed))
    o = ro.OracleRod(c["n"], c["init"][0:3], c["init"][3:6], c["init"][6:9], c["L"], c["r"], c["rho"], c["E"], c["dt"],
                     gravity=c["g"], damping_constant=c["damping"], bc_kind=c["bc"])
    o.substeps(300)
    assert np.isfinite(o.position_collection).all(), "unstable random case (test generator problem)"
    names = ("position_collection", "velocity_collection", "director_collection", "omega_collection")
    mk = lambda: ro.OracleRod(c["n"], c["init"][0:3], c["init"][3:6], c["init"][6:9], c["L"], c["r"], c["rho"], c["E"], c["dt"],
                              gravity=c["g"], damping_constant=c["damping"], bc_kind=c["bc"])
    sens = one_ulp_divergence(mk, lambda rod: rod.substeps(300), {k: getattr(o, k).copy() for k in names})
    for math in (nat.MATH_FAST, nat.MATH_FAITHFUL):
        h = nat.Handle(model=nat.MODEL_ROD, n_env=3, n_elem=c["n"], dt=c["dt"], base_length=c["L"], base_radius=c["r"],
                       density=c["rho"], youngs_modulus=c["E"], gravity=tuple(c["g"]), damping_constant=c["damping"],
                       bc_kind=c["bc"], math=math)
        h.reset_host(np.repeat(c["init"][None, :], 3, axis=0))
        h.step_host(None, 120); h.step_host(None, 180)
        f = {k: v.cpu().numpy() for k, v in h.fields().items()}
        floors = rate_floors(c["E"], c["rho"], c["L"], c["n"], c["r"], np.abs(o.position_collection).max())
        for name in ("position_collection", "velocity_collection", "director_collection", "omega_collection"):
            assert_state_close(f[name][1], getattr(o, name), name, floors, f"seed={seed} math={math} n={c['n']} bc={c['bc']}", measured=sens)
        h.close()


def test_continuum_snake_env_golden_first_steps(golden_dir):
    """§8 f2: ContinuumSnake-v0 — travelling-wave MuscleTorques + anisotropic plane friction, 25 000
    substeps per env-step — through the Gymnasium facade vs the reference-env-on-shim fixture.

    This env has kinetic friction only, regularised over |v| in [1e-8, 2e-8] m/s and integrated
    explicitly with dt mu g / tol ~ 1e3: wherever the rod sticks sideways the reference itself
    chatters with amplitude a = dt * 2 mu g ~ 1.4e-5 m/s (and a / r ~ 4e-3 rad/s in roll), with a
    round-off dependent phase.  Without friction the same kernel path agrees with the shim to 1e-11
    (DESIGN.md 5); with it, two correct implementations agree to a few chatter amplitudes, which is
    what the bounds below are (measured: 2.3e-7 m, 2.4e-5 m/s, 1.4e-5, 5.6e-3 rad/s)."""
    import gym_softrobot_b200 as gsb
    g = np.load(os.path.join(golden_dir, "continuum_snake_seed42.npz"))
    env = gsb.make("ContinuumSnake-v0")
    assert env.step_skip == int(g["step_skip"]) == 25000
    obs0, _ = env.reset(seed=42)
    assert obs0.dtype == np.float32 and obs0.shape == (756,)
    np.testing.assert_array_equal(obs0, g["obs0"])
    bounds = {"position": 1e-6, "velocity": 1e-4, "director": 5e-5, "omega": 3e-2}   # absolute
    n_state = sum(1 for k in g.files if k.startswith("beta"))
    for i in range(n_state):
        obs, r, te, tr, info = env.step(g["actions"][i])
        assert env.time == float(g["time"][i])                 # the in-kernel clock, bit for bit
        st = env.rod_state()
        for gk, tol in bounds.items():
            err = float(np.abs(st[FIELDS[gk]] - g[f"state{i + 1}/{gk}"]).max())
            assert err < tol, f"step {i} field {gk} abs err {err:.3e}"
        np.testing.assert_allclose(obs[:306], g[f"obs{i + 1}"][:306], rtol=0, atol=1e-4)    # x, v
        np.testing.assert_allclose(obs[306:], g[f"obs{i + 1}"][306:], rtol=0, atol=5e-5)    # Q
        assert r == 0.0 == float(g["reward"][i]) and (te, tr) == (False, False)
    env.close()


def test_continuum_snake_long_horizon_is_a_replica_of_the_reference(golden_dir):
    """33 env-steps (825 000 substeps, 6.6 s): the chatter above makes the trajectory sensitive — GPU
    runs whose initial node positions differ by 1e-15 m drift apart by 4e-8 m (0.2 s), 3e-5 m (2 s),
    4e-3 m (6.6 s) in the centre of mass.  Parity criterion for such a system: the reference run must be
    indistinguishable from one more perturbed replica.  Eight envs (one exact, seven perturbed) are
    stepped with the fixture's actions; at every callback sample the reference's centre of mass must lie
    within 4x the replicas' own spread, and every reward within 4 sigma of the replicas' rewards."""
    import torch
    import gym_softrobot_b200 as gsb
    g = np.load(os.path.join(golden_dir, "continuum_snake_seed42.npz"))
    N = 8
    v = gsb.make_vec("ContinuumSnake-v0", N, autoreset=False)
    v.reset()
    x = v.handle.fields()["position_collection"]
    noise = 1e-15 * torch.randn(x.shape, device="cuda", dtype=torch.float64,
                                generator=torch.Generator(device="cuda").manual_seed(1))
    noise[0] = 0
    x += noise
    rewards = []
    for i, a in enumerate(g["actions"]):
        obs, r, te, tr, info = v.step(torch.as_tensor(a, device="cuda")[None].repeat(N, 1))
        rewards.append(r.cpu().numpy())
        assert float(info["time"][0]) == float(g["time"][i])
        assert not bool(te.any()) and bool(tr.any()) == bool(g["truncated"][i])
    rewards = np.array(rewards)                                   # [33, N]
    S = len(g["cb_time"])
    assert len(v._times) == S and np.array_equal(np.array(v._times), g["cb_time"])
    com, vel = v._com[:, :S].cpu().numpy(), v._vel[:, :S].cpu().numpy()
    for arr, ref, floor in ((com, g["cb_com"], 1e-7), (vel, g["cb_avg_velocity"], 5e-6)):
        spread = np.abs(arr[1:] - arr[:1]).max(axis=(0, 2))       # replicas vs the exact run, per sample
        dev = np.abs(arr[0] - ref).max(axis=1)
        worst = float((dev / (4 * spread + floor)).max())
        assert worst < 1.0, f"reference outside the replicas' spread by {worst:.2f}x"
    assert np.all(rewards[g["reward"] == 0.0] == 0.0)             # no reward before three periods
    nz = g["reward"] != 0.0
    assert nz.sum() >= 3
    mean, std = rewards[nz].mean(axis=1), rewards[nz].std(axis=1)
    assert np.all(np.abs(g["reward"][nz] - mean) < 4 * std + 1e-6), (g["reward"][nz], mean, std)
    assert np.all(std < 0.05 * np.abs(mean))                      # and the spread itself is a few per cent
    # the reference drifts from ITSELF by the same amounts: its own 1e-15-perturbed replica (second fixture) is as far
    # from the reference run as the GPU replicas are from each other, and passes the same two checks
    p = np.load(os.path.join(golden_dir, "continuum_snake_seed42_perturbed.npz"))
    own = np.abs(p["cb_com"] - g["cb_com"]).max(axis=1)
    gpu_spread = np.abs(com[1:] - com[:1]).max(axis=(0, 2))
    for k in (12, 36, 120, 240, S - 1):
        assert 0.1 * gpu_spread[k] < own[k] < 10 * gpu_spread[k] + 1e-7, (k, own[k], gpu_spread[k])
    assert np.all(np.abs(p["reward"][nz] - mean) < 4 * std + 1e-6)
    v.close()


@pytest.mark.parametrize("mode", [1, 2], ids=["fixed-target", "moving-target"])
def test_soft_arm_tracking_env_golden(golden_dir, mode):
    """§8 f4 (spline muscle actuation): SoftArmTracking-v0 — clamped arm, two
    MuscleTorquesWithVaryingBetaSplines forcings re-fitted in-kernel at the current element lengths —
    through the Gymnasium facade vs the reference-env-on-shim fixture (40 env-steps of 50 substeps,
    float64 observations; steps 4-5 repeat an action so the cached torque profile path is exercised)."""
    import gym_softrobot_b200 as gsb
    g = np.load(os.path.join(golden_dir, f"soft_arm_tracking_mode{mode}_seed42.npz"))
    env = gsb.make("SoftArmTracking-v0", game_mode=mode)
    obs0, _ = env.reset(seed=42)
    assert obs0.dtype == np.float64 and obs0.shape == (14,)
    np.testing.assert_allclose(obs0, g["obs0"], rtol=0, atol=1e-15)
    for i, a in enumerate(g["actions"]):
        obs, r, te, tr, info = env.step(a)
        if f"state{i + 1}/position" in g.files:
            st = env.rod_state()
            for gk in ("position", "velocity", "director", "omega", "kappa"):
                err = rel(st[FIELDS[gk]], g[f"state{i + 1}/{gk}"])
                assert err < 1e-9, f"step {i} field {gk} rel err {err:.3e}"
        np.testing.assert_allclose(obs, g["obs"][i], rtol=1e-9, atol=1e-12)
        assert abs(r - float(g["reward"][i])) < 1e-9
        assert (te, tr) == (bool(g["terminated"][i]), bool(g["truncated"][i]))
        assert info["ctime"] == float(g["ctime"][i])
    env.close()


def test_octo_flat_decentralized_mode_golden(golden_dir):
    """FlatEnv(policy_mode="decentralized") (flat_env.py:111-145,248-260): per-arm action space, one action
    row per arm, one-hot arm id appended to every row of the individual observation."""
    import gym_softrobot_b200 as gsb
    g = np.load(os.path.join(golden_dir, "octo_flat_decentralized_seed42.npz"))
    env = gsb.make("OctoFlat-v0", recording_fps=int(g["recording_fps"]), policy_mode="decentralized")
    assert env.action_space.shape == tuple(g["action_shape"]) == (3,)
    obs0, _ = env.reset(seed=42)
    assert obs0["individual"].shape == g["obs0/individual"].shape == (8, 64)
    np.testing.assert_allclose(obs0["individual"], g["obs0/individual"], rtol=1e-6, atol=1e-7)
    np.testing.assert_array_equal(obs0["individual"][:, -8:], np.eye(8, dtype=np.float32))
    obs, r, te, tr, info = env.step(g["action"])                 # [n_arm, n_action]
    np.testing.assert_allclose(obs["individual"], g["obs1/individual"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(obs["shared"], g["obs1/shared"], rtol=1e-4, atol=1e-6)
    assert abs(r - float(g["reward"])) < 1e-6 and not te and not tr
    env.close()


@pytest.mark.parametrize("v0,mu", [(0.1, 0.2), (-0.1, 0.3)], ids=["forward", "backward"])
def test_sliding_rod_decelerates_at_mu_g_on_gpu(v0, mu):
    """The Coulomb-friction known answer of tests/test_oracle_golden.py on the CUDA path: a rod sliding along
    its axis slows down at mu_kinetic * g when the contact runs after gravity (the envs' order) and not at
    all when it runs before."""
    import torch
    nat = _native()
    g, dt, steps, r = 9.81, 1e-5, 2000, 0.01
    for before in (False, True):
        c = dict(plane_origin=[0.0, 0.0, -r], plane_normal=[0.0, 0.0, 1.0], k=1e2, nu=1e1, slip_velocity_tol=1e-8,
                 static_mu=[0.4, 0.6, 0.8], kinetic_mu=[0.2, 0.3, 0.4], before_forcing=before)
        h = nat.Handle(model=nat.MODEL_ROD, n_env=4, n_elem=20, dt=dt, base_length=1.0, base_radius=r, density=1000.0,
                       youngs_modulus=1e6, gravity=(0.0, 0.0, -g), bc_kind=nat.BC_FREE, contact=c)
        init = np.zeros((4, 9)); init[:, 3] = 1.0; init[:, 8] = 1.0
        h.reset_host(init)
        h.fields()["velocity_collection"][:, 0, :] = v0
        h.step_host(None, steps)
        v = h.fields()["velocity_collection"][:, 0, :].cpu().numpy()
        expected = v0 if before else v0 - np.sign(v0) * mu * g * dt * steps
        assert np.abs(v - expected).max() < 1e-3 * abs(v0)
        h.close()


def test_spline_torque_forcing_rate_limited_and_tangent(golden_dir):
    """The spline-torque ABI beyond what SoftArmTracking-v0 uses: finite max_rate (the cached control values
    creep towards the targets by 0.04 per substep, each time re-fitting the spline at the current lengths),
    twist (tangent) direction, 3 control points — against the reference's forcing class driven directly on
    the shim rod (oracle/gen_golden.py:gen_spline_forcing)."""
    import torch
    nat = _native()
    g = np.load(os.path.join(golden_dir, "spline_forcing_seed5.npz"))
    n, seg = int(g["n_elem"]), int(g["segment"])
    h = nat.Handle(model=nat.MODEL_ROD, n_env=3, n_elem=n, dt=float(g["dt"]), base_length=float(g["base_length"]),
                   base_radius=float(g["base_radius"]), density=1000.0, youngs_modulus=float(g["youngs_modulus"]),
                   damping_constant=float(g["damping_constant"]), bc_kind=nat.BC_ONE_END_FIXED,
                   spline=dict(directions=(0, 2), n_ctrl=int(g["n_ctrl"]), scale=float(g["scale"]), max_rate=float(g["max_rate"])))
    init = np.zeros((3, 9)); init[:, 5] = 1.0; init[:, 6] = 1.0          # direction +z, normal +x
    h.reset_host(init)
    pts, mags = h.spline_tensors()
    for s, tgt in enumerate(g["targets"]):
        pts[:, 0, :3] = torch.as_tensor(tgt[0], device="cuda")
        pts[:, 2, :3] = torch.as_tensor(tgt[1], device="cuda")
        h.step_host(None, seg)
        f = {k: v.cpu().numpy() for k, v in h.fields().items()}
        for gk in ("position", "velocity", "director", "omega", "kappa"):
            for e in range(3):
                err = rel(f[FIELDS[gk]][e], g[f"seg{s + 1}/{gk}"])
                assert err < 1e-9, f"segment {s} field {gk} rel err {err:.3e}"
    # 50 substeps at 0.04 per substep cover a change of (just about) 2: the cached values are at the targets
    assert torch.allclose(pts[:, 0, 3:6], pts[:, 0, :3], rtol=0, atol=0.05) and float(mags[:, 1].abs().max()) == 0.0
    h.close()


@pytest.mark.parametrize("case", ["A", "B"], ids=["frictionless-plane", "free-oblique-phase"])
def test_muscle_torques_without_friction_are_roundoff_limited(golden_dir, case):
    """The travelling-wave `MuscleTorques` path at full precision: the snake rod without friction (A: plane
    with zero friction coefficients + gravity; B: no plane, oblique torque direction, phase shift), forcing
    rebuilt half way like `set_action` does.  3000 substeps, 1e-9 — the statistical criterion of the
    ContinuumSnake tests is needed for the friction law only."""
    import torch
    from gym_softrobot_b200.envs.snake import snake_contact_params, beta_spline_matrix
    nat = _native()
    g = np.load(os.path.join(golden_dir, "muscle_torques_seed9.npz"))
    n, L, E = int(g["n_elem"]), 0.35, 1e6
    contact = None
    if case == "A":
        contact = snake_contact_params()
        contact["kinetic_mu"] = np.zeros(3)
    h = nat.Handle(model=nat.MODEL_ROD, n_env=2, n_elem=n, dt=float(g["dt"]), base_length=L, base_radius=L * 0.011,
                   density=1000.0, youngs_modulus=E, shear_modulus=E / 1.5, damping_constant=1e-4,
                   gravity=(0.0, -9.80665, 0.0) if case == "A" else (0.0, 0.0, 0.0), contact=contact,
                   muscle=dict(period=float(g["period"]), ramp_up_time=float(g["period"]), phase_shift=float(g[f"{case}/phase"]),
                               direction=g[f"{case}/direction"]))
    init = np.zeros((2, 9)); init[:, 5] = 1.0; init[:, 7] = 1.0
    h.reset_host(init)
    mu = h.muscle_tensor()
    W = beta_spline_matrix(6, n)
    # measured conditioning of this very configuration (the rod hardly moves in 12-24 ms and, in case A, rests on a stiff
    # contact spring): the C oracle run three times — as is, from a one-ulp different start, built with FMA contraction
    import rod_oracle as ro
    names = ("position_collection", "velocity_collection", "director_collection", "omega_collection")
    mus = dict(period=float(g["period"]), ramp_up_time=float(g["period"]), phase_shift=float(g[f"{case}/phase"]), direction=g[f"{case}/direction"])
    def make():
        return ro.OracleRod(n, [0, 0, 0], [0, 0, 1.0], [0, 1.0, 0], L, L * 0.011, 1000.0, E, float(g["dt"]), shear_modulus=E / 1.5,
                            damping_constant=1e-4, gravity=(0.0, -9.80665, 0.0) if case == "A" else (0.0, 0.0, 0.0), contact=contact, muscle=mus)
    def advance(rod, upto):
        for k in range(upto + 1):
            rod.muscle[0] = float(g[f"{case}/wave_number{k}"]); rod.muscle[1:] = W @ g[f"{case}/b{k}"].astype(np.float64)
            rod.substeps(int(g["segment"]))
    for seg in range(2):
        beta = W @ g[f"{case}/b{seg}"].astype(np.float64)
        np.testing.assert_allclose(beta, g[f"{case}/beta{seg}"], rtol=0, atol=1e-17)
        mu[:, 2:] = torch.as_tensor(beta, device="cuda")
        mu[:, 1] = float(g[f"{case}/wave_number{seg}"])
        h.step_host(None, int(g["segment"]))
        f = {k: v.cpu().numpy() for k, v in h.fields().items()}
        floors = rate_floors(E, 1000.0, L, n, L * 0.011, L)      # the rod hardly moves in 12-24 ms: see rate_floors
        o = make(); advance(o, seg)
        ref = {k: getattr(o, k).copy() for k in names}
        s1, s2 = one_ulp_divergence(make, lambda rod: advance(rod, seg), ref), fma_build_divergence(make, lambda rod: advance(rod, seg), ref)
        sens = {k: max(s1[k], s2[k]) for k in names}
        o.close()
        for gk in ("position", "velocity", "director", "omega"):
            assert_state_close(f[FIELDS[gk]][1], g[f"{case}/seg{seg + 1}/{gk}"], FIELDS[gk], floors, f"case {case} segment {seg}", measured=sens)
    assert float(mu[0, 0]) == float(g[f"{case}/time"])
    h.close()


def test_fast_only_kernel_falls_back_per_env():
    """The default path is a fast-only kernel (no warp-vote fallbacks in the substep body) followed by the
    safe kernel over the envs the first one flagged.  Here two of six free rods spin so fast that the half-step
    rotation leaves the polynomial range (|h w| = 1 rad per half step: q = 1 > 0.25) and a third carries a
    30 degree kink between two elements (outside the narrow bend map), so they must be
    re-run by the fallback with libm-class accuracy while the others stay on the fast path; every env is
    compared with the oracle, twice in a row (the flags must have been cleared).  Only 20 substeps in all: a rod
    spinning at 2e4 rad/s amplifies round-off exponentially (7e-9 after 20 substeps, O(1) after 50, in the safe
    single-kernel path exactly as in this one — their results are bit-identical)."""
    import torch
    import rod_oracle as ro
    nat = _native()
    n_env, n, dt, radius = 6, 30, 1e-4, 0.05
    init = _tilted_init(n_env)
    kw = dict(density=1000.0, youngs_modulus=1e6)
    h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n, dt=dt, base_length=1.0, base_radius=radius,
                   gravity=(0.0, -9.80665, 0.0), damping_constant=2e-3, bc_kind=nat.BC_FREE, **kw)
    h.reset_host(init)
    rods = [ro.OracleRod(n, init[i, 0:3], init[i, 3:6], init[i, 6:9], 1.0, radius, 1000.0, 1e6, dt,
                         gravity=(0.0, -9.80665, 0.0), damping_constant=2e-3) for i in range(n_env)]
    spin = np.zeros((n_env, 3, n))
    spin[1, 2, :] = 2.0e4                     # rigid spin about the rod axis (d3): no strain, huge rotation per substep
    spin[4, 2, :] = -2.0e4
    h.fields()["omega_collection"][:] = torch.as_tensor(spin, device="cuda")
    for i, r in enumerate(rods):
        r.omega_collection[:] = spin[i]
    # env 2: a 30 degree kink between elements 14 and 15 (u = sin^2(15 deg) = 0.067 > 0.04): the bend map's range
    kink = np.deg2rad(30.0)
    Rk = np.array([[np.cos(kink), np.sin(kink), 0.0], [-np.sin(kink), np.cos(kink), 0.0], [0.0, 0.0, 1.0]])
    Q2 = rods[2].director_collection.copy()
    for k in range(15, n):
        Q2[:, :, k] = Rk @ Q2[:, :, k]           # rotate the frames of the outer half about d3
    rods[2].director_collection[:] = Q2
    h.fields()["director_collection"][2] = torch.as_tensor(Q2, device="cuda")
    for chunk in (8, 12):
        obs, rew, term = h.step_host(None, chunk)
        f = {k: v.cpu().numpy() for k, v in h.fields().items()}
        for i, r in enumerate(rods):
            r.substeps(chunk)
            floors = rate_floors(1e6, 1000.0, 1.0, n, radius, np.abs(r.position_collection).max())
            for name in ("position_collection", "velocity_collection", "director_collection", "omega_collection"):
                assert_state_close(f[name][i], getattr(r, name), name, floors, f"env {i}")
        assert term.sum() == 0
    assert h.launch_count >= 1 + 2 * 2        # reset + (fast-only, fallback) per step
    h.close()


def test_fast_pair_switches_itself_off_when_most_envs_fall_back():
    """Adaptive switch of the fast-only / fallback pair: a handle whose envs all live outside the narrow fast-math
    range (here: every rod spins at 3000 rad/s, 0.15 rad per half-step rotation > 0.1) would pay for two
    kernels per step; after the first asynchronous check of the fallback counter (steps 8-16) it must be down to
    the single safe kernel.  A well-behaved handle next to it keeps the pair."""
    import torch
    nat = _native()
    n_env, n = 8, 20

    def make(spin):
        h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n, dt=1e-4, base_length=1.0, base_radius=0.05,
                       density=1000.0, youngs_modulus=1e6, gravity=(0.0, -9.80665, 0.0), damping_constant=2e-3)
        h.reset_host(_tilted_init(n_env))
        if spin:
            h.fields()["omega_collection"][:, 2, :] = 3000.0
        return h

    for spin, per_step_late in ((True, 1), (False, 2)):
        h = make(spin)
        counts = []
        for _ in range(110):
            h.step_host(None, 1)
            counts.append(h.launch_count)
        assert counts[0] - 1 == 2                                    # reset + (fast-only, fallback)
        late = np.diff(counts[-10:])
        assert np.all(late == per_step_late), (spin, late)
        assert torch.isfinite(h.state_tensor()).all()
        h.close()


def test_newton_reciprocals_are_one_ulp():
    """rsqrt_nr / rcp_nr (MUFU seed + one third-order Newton step, csrc/rod_math.cuh) against the correctly rounded
    IEEE results over 2^20 log-spaced arguments spanning the lengths / dilatations the kernels see and far beyond."""
    nat = _native()
    e_rsqrt, e_rcp = nat.selftest_reciprocals(1 << 20, 1e-12, 1e12)
    assert 0.0 < e_rsqrt < 3.4e-16 and 0.0 < e_rcp < 2.3e-16, (e_rsqrt, e_rcp)   # <= 1.5 ulp / <= 1 ulp


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_muscle_torques_vs_c_oracle_randomized(seed):
    """Travelling-wave muscle torques at parameters no fixture holds: rod size, wave number, phase, direction and
    beta profile drawn per seed, CUDA path vs the C oracle's own restatement (free rod, no friction), 1e-9."""
    import torch
    import rod_oracle as ro
    nat = _native()
    rng = np.random.default_rng(100 + seed)
    n = int(rng.integers(12, 60)); L = float(rng.uniform(0.2, 0.6)); r0 = L * float(rng.uniform(0.008, 0.02))
    E, rho, dt, period = 1e6, 1000.0, 8e-6, float(rng.uniform(1.0, 3.0))
    direction = rng.standard_normal(3); direction /= np.linalg.norm(direction)
    mus = dict(period=period, ramp_up_time=0.5 * period, phase_shift=float(rng.uniform(0, 6.28)), direction=direction)
    beta = rng.uniform(-4e-3, 4e-3, n) * np.sin(np.linspace(0, np.pi, n))
    kw = float(rng.uniform(3.0, 12.0))
    init = np.zeros((2, 9)); init[:, 5] = 1.0; init[:, 7] = 1.0
    h = nat.Handle(model=nat.MODEL_ROD, n_env=2, n_elem=n, dt=dt, base_length=L, base_radius=r0, density=rho,
                   youngs_modulus=E, shear_modulus=E / 1.5, damping_constant=1e-4, muscle=mus)
    h.reset_host(init)
    mu = h.muscle_tensor()
    mu[:, 1] = kw
    mu[:, 2:] = torch.as_tensor(beta, device="cuda")
    o = ro.OracleRod(n, [0, 0, 0], [0, 0, 1.0], [0, 1.0, 0], L, r0, rho, E, dt, shear_modulus=E / 1.5,
                     damping_constant=1e-4, muscle=mus)
    o.muscle[0] = kw; o.muscle[1:] = beta
    for chunk in (700, 800):
        h.step_host(None, chunk); o.substeps(chunk)
        f = {k: v.cpu().numpy() for k, v in h.fields().items()}
        floors = rate_floors(E, rho, L, n, r0, L)
        for name in ("position_collection", "velocity_collection", "director_collection", "omega_collection"):
            assert_state_close(f[name][1], getattr(o, name), name, floors, f"seed {seed}")
    assert float(mu[0, 0]) == o.time
    h.close(); o.close()


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_spline_torques_vs_c_oracle_randomized(seed):
    """Spline muscle torques at parameters no fixture holds (rod size, number of control points, directions, rate
    limit, scale drawn per seed; targets changed every 40 substeps): CUDA path vs the C oracle's independent
    restatement of the reference forcing, clamped rod, 1e-9."""
    import torch
    import rod_oracle as ro
    nat = _native()
    rng = np.random.default_rng(200 + seed)
    n = int(rng.integers(10, 64)); L = float(rng.uniform(0.3, 1.5)); r0 = L / n * float(rng.uniform(0.5, 1.2))
    E, rho, dt = 1e6, 1000.0, 2e-5
    P = int(rng.integers(2, 7))
    dirs = tuple(sorted(rng.choice(3, size=int(rng.integers(1, 4)), replace=False).tolist()))
    EI = E * np.pi * r0 ** 4 / 4
    spl = dict(directions=dirs, n_ctrl=P, scale=float(EI * rng.uniform(0.5, 3.0)), max_rate=float(rng.uniform(0.02, 0.2)))
    init = np.zeros((2, 9)); init[:, 5] = 1.0; init[:, 6] = 1.0
    h = nat.Handle(model=nat.MODEL_ROD, n_env=2, n_elem=n, dt=dt, base_length=L, base_radius=r0, density=rho,
                   youngs_modulus=E, damping_constant=0.5, bc_kind=nat.BC_ONE_END_FIXED, spline=spl)
    h.reset_host(init)
    o = ro.OracleRod(n, [0, 0, 0], [0, 0, 1.0], [1.0, 0, 0], L, r0, rho, E, dt, damping_constant=0.5,
                     bc_kind=ro.BC_ONE_END_FIXED, spline=spl)
    pts, mags = h.spline_tensors()
    for seg in range(6):
        tgt = rng.uniform(-1, 1, (3, P))
        for d in dirs:
            pts[:, d, :P] = torch.as_tensor(tgt[d], device="cuda")
            o.spline_points[d, :P] = tgt[d]
        h.step_host(None, 40); o.substeps(40)
        f = {k: v.cpu().numpy() for k, v in h.fields().items()}
        floors = rate_floors(E, rho, L, n, r0, L)
        for name in ("position_collection", "velocity_collection", "director_collection", "omega_collection"):
            assert_state_close(f[name][1], getattr(o, name), name, floors, f"seed {seed} seg {seg}")
        for d in dirs:
            np.testing.assert_allclose(mags[1, d].cpu().numpy(), o.spline_magnitude[d], rtol=1e-9, atol=1e-12 * spl["scale"])
    h.close(); o.close()


def test_octo_cfg4_8x40_vs_reference_fixture(golden_dir):
    """BASELINE config 4 as specified — build_octopus(n_arm=8, n_elem=40) (envs/octopus/build.py:52-217) under
    FlatEnv actuation — at the dt that is stable for 40 elements (3e-5), 3 x 333 = 999 substeps, every field
    (kappa, sigma, dilatation included) at 1e-9 against the fixture the reference's own env / joint / constraint
    code produced on the shim (oracle/gen_golden.py:gen_octo_cfg4)."""
    import gym_softrobot_b200 as gsb
    g = np.load(os.path.join(golden_dir, "octo_cfg4_8x40_seed42.npz"))
    env = gsb.make("OctoFlat-v0", n_elems=int(g["n_elems"]), time_step=float(g["time_step"]),
                   recording_fps=int(g["recording_fps"]))
    assert env.step_skip == int(g["step_skip"]) == 333
    env.reset(seed=42)
    np.testing.assert_allclose(env._target, g["target"], rtol=0, atol=0)
    worst = 0.0
    for i, a in enumerate(g["actions"]):
        obs, r, te, tr, info = env.step(a)
        st = env.state()
        # the host-side interpolation matrix reproduces what the reference's set_action wrote
        rk = env._vec.handle.rest_kappa_tensor().cpu().numpy()
        assert np.abs(rk - g["rest_kappa"][i]).max() < 1e-12 * np.abs(g["rest_kappa"][i]).max()
        for arm in range(8):
            for gk, fk in FIELDS.items():
                err = _asm_err(st[fk][arm], g[f"state{i + 1}/arm{arm}/{gk}"], fk)
                worst = max(worst, err)
                assert err < TOL, f"step {i} arm {arm} {gk}: {err:.3e}"
        hd = st["head"]
        for sl, gk, fk in ((slice(0, 3), "position", "position_collection"), (slice(3, 6), "velocity", "velocity_collection"),
                           (slice(6, 15), "director", "director_collection"), (slice(15, 18), "omega", "omega_collection")):
            err = _asm_err(hd[sl], g[f"state{i + 1}/head/{gk}"].reshape(-1), fk)
            worst = max(worst, err)
            assert err < TOL, f"step {i} head {gk}: {err:.3e}"
        assert abs(r - float(g["reward"][i])) < 1e-6 and te == bool(g["terminated"][i])
    print(f"cfg4 8x40 vs reference fixture: worst {worst:.2e}")
    env.close()


def _random_assembly(seed, friction_multiplier):
    """Per-seed assembly parameters + a factory of the multi-rod C oracle for them."""
    import rod_oracle as ro
    rng = np.random.default_rng(1000 + seed)
    n_arm = int(rng.integers(2, 9))
    n_elem = [8, 10, 13, 20, 31, 40][seed]   # every seed a different element count, 40 (config 4) included
    L0, r0 = 0.35, 0.35 * 0.02
    p = dict(n_arm=n_arm, n_elem=n_elem, head_radius=float(rng.uniform(0.03, 0.06)), head_density=float(rng.uniform(300, 900)),
             kt=float(10 ** rng.uniform(-1, 2)), nu=float(10 ** rng.uniform(-4, -2)))
    # explicit stability of the joint spring on the half-mass end node: dt < 2 sqrt(m / k), keep a factor 3
    m_end = 0.5 * 1000.0 * np.pi * r0 * r0 * L0 / n_elem
    p["k"] = float(10 ** rng.uniform(4.5, 6))
    p["dt"] = float(min(7e-5, 2 * np.sqrt(m_end / p["k"]) / 3, 0.25 * (L0 / n_elem) / np.sqrt(1e6 / 1000.0)))
    s = np.linspace(0, 1, n_elem - 1)
    p["rest_kappa"] = []          # smooth random rest curvature about d1 and a little about d2, per chunk and arm
    for chunk in range(3):
        rk = np.zeros((n_arm, 3, n_elem - 1))
        for a in range(n_arm):
            rk[a, 0] = rng.uniform(-12, 12) * np.sin(np.pi * s) + rng.uniform(-6, 6) * np.sin(2 * np.pi * s)
            rk[a, 1] = rng.uniform(-3, 3) * np.sin(np.pi * s)
        p["rest_kappa"].append(rk)

    def make_oracle():
        return ro.octopus_assembly(n_arm=n_arm, n_elem=n_elem, time_step=p["dt"], head_radius=p["head_radius"],
                                   head_density=p["head_density"], body_arm_k=p["k"], body_arm_kt=p["kt"],
                                   body_arm_nu=p["nu"], friction_multiplier=friction_multiplier)
    return p, make_oracle


def _oracle_states(asm, p):
    out = []
    for rk in p["rest_kappa"]:
        for a, rod in enumerate(asm.arms):
            rod.rest_kappa[...] = rk[a]
        asm.substeps(300)
        st = {fk: np.stack([getattr(rod, fk).copy() for rod in asm.arms]) for fk in FIELDS.values()}
        st["head"] = np.concatenate([asm.head_position, asm.head_velocity, asm.head_director.reshape(-1), asm.head_omega])
        out.append(st)
    return out


HEAD_SLICES = ((slice(0, 3), "position_collection"), (slice(3, 6), "velocity_collection"),
               (slice(6, 15), "director_collection"), (slice(15, 18), "omega_collection"))


@pytest.mark.parametrize("friction", [False, True], ids=["frictionless-plane", "friction"])
@pytest.mark.parametrize("seed", [0, 1, 2, 3, 4, 5])
def test_randomized_assembly_vs_c_oracle(seed, friction):
    """Arms + rigid head + FixedJoint2Rigid + BodyBoundaryCondition on the plane with per-seed arm count, element
    count, joint stiffness / damping / torsional stiffness, head size and density and per-arm rest curvature, against
    the multi-rod C oracle (oracle/rod_oracle.c: ro_assembly), every field, 900 substeps.

    frictionless-plane (normal response, gravity, joints, head, BC all active): 1e-9 throughout.
    friction: 1e-9 as well once the arms move (chunks 2 and 3, 600 substeps).  The start from rest is different: with
    every velocity inside the friction law's regularisation band (|v| in [1e-8, 2e-8] m/s, integrated explicitly with
    dt mu g / tol >> 2) the model amplifies round-off by 1e7 within 60 substeps — the ORACLE ITSELF, restarted with its
    velocities perturbed by 1e-12 m/s, moves by 1e-5 m/s in chunk 1 and not at all (2.6e-12) in chunks 2 and 3
    (measured, seeds 2-5).  Chunk 1 is therefore bounded by 20 x the largest divergence among three perturbed oracle
    replicas (calibrated on the spot, never below 1e-9), after which the CUDA state is re-synchronised with the oracle's."""
    import torch
    nat = _native()
    p, make_oracle = _random_assembly(seed, 1.0 if friction else 0.0)
    n_arm, n_elem, dt = p["n_arm"], p["n_elem"], p["dt"]
    asm = make_oracle()
    ref = _oracle_states(asm, p)
    asm.close()
    bound = [{fk: TOL for fk in list(FIELDS.values()) + ["head"]} for _ in ref]
    if friction:
        for rep in range(3):
            asm = make_oracle()
            prng = np.random.default_rng(77 + rep)
            for rod in asm.arms:      # what "another correct implementation" looks like after a few substeps
                rod.velocity_collection[...] += 1e-12 * prng.standard_normal(rod.velocity_collection.shape)
            st = _oracle_states(asm, dict(p, rest_kappa=p["rest_kappa"][:1]))[0]
            for fk in FIELDS.values():
                bound[0][fk] = max(bound[0][fk], 20 * max(_asm_err(st[fk][a], ref[0][fk][a], fk) for a in range(n_arm)))
            bound[0]["head"] = max(bound[0]["head"], 20 * max(_asm_err(st["head"][sl], ref[0]["head"][sl], fk) for sl, fk in HEAD_SLICES))
            asm.close()
    from gym_softrobot_b200.envs.arm_single import arm_contact_params, _ROD, _G
    n_env, r0 = 3, 0.35 * 0.02
    h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n_elem, dt=dt, gravity=(0.0, 0.0, _G), damping_constant=1e-2,
                   bc_kind=nat.BC_FREE, contact=arm_contact_params(friction_multiplier=1.0 if friction else 0.0), n_rod=n_arm,
                   head=dict(length=2 * r0, radius=p["head_radius"], density=p["head_density"]),
                   joint=dict(radius=p["head_radius"], angles_deg=[360 / n_arm * a for a in range(n_arm)], k=p["k"], nu=p["nu"], kt=p["kt"]),
                   **_ROD)
    row = []
    for a in range(n_arm):
        c, s = np.cos(np.deg2rad(360 / n_arm * a)), np.sin(np.deg2rad(360 / n_arm * a))
        row += [c * p["head_radius"], s * p["head_radius"], 0.0, c, s, 0.0, 0.0, 0.0, 1.0]
    row += [0.0, 0.0, -r0, 0.0, 0.0, 1.0, 0.0, 1.0, 0.0]
    h.reset(torch.as_tensor(np.repeat(np.array([row]), n_env, axis=0), device="cuda").contiguous())
    o6 = torch.empty((n_env, 6), dtype=torch.float32, device="cuda")
    rew = torch.empty(n_env, dtype=torch.float64, device="cuda")
    term = torch.empty(n_env, dtype=torch.uint8, device="cuda")
    worst, worst_ratio = 0.0, 0.0
    for chunk, rk in enumerate(p["rest_kappa"]):
        h.rest_kappa_tensor().unflatten(0, (n_env, n_arm))[:] = torch.as_tensor(rk, device="cuda")
        h.step(None, 300, o6, rew, term)
        f = {k_: v.cpu().numpy() for k_, v in h.fields().items()}
        hd = h.head_tensor().cpu().numpy()
        assert int(term.sum()) == 0
        for e in range(n_env):
            for a in range(n_arm):
                for fk in FIELDS.values():
                    err = _asm_err(f[fk][e, a], ref[chunk][fk][a], fk)
                    worst, worst_ratio = max(worst, err), max(worst_ratio, err / bound[chunk][fk])
                    assert err < bound[chunk][fk], (f"seed {seed} (n_arm {n_arm}, n_elem {n_elem}, k {p['k']:.2e}) chunk {chunk} env {e} "
                                                     f"arm {a} {fk}: {err:.3e} (bound {bound[chunk][fk]:.1e})")
            for sl, fk in HEAD_SLICES:
                err = _asm_err(hd[e, sl], ref[chunk]["head"][sl], fk)
                worst, worst_ratio = max(worst, err), max(worst_ratio, err / bound[chunk]["head"])
                assert err < bound[chunk]["head"], f"seed {seed} chunk {chunk} head {fk}: {err:.3e} (bound {bound[chunk]['head']:.1e})"
        if friction and chunk == 0:
            # re-synchronise after the chaotic start from rest: the oracle's state goes into the CUDA handle
            fl = h.fields()
            for fk in ("position_collection", "velocity_collection", "director_collection", "omega_collection"):
                fl[fk][:] = torch.as_tensor(ref[0][fk], device="cuda")
            h.head_tensor()[:, :18] = torch.as_tensor(ref[0]["head"], device="cuda")
            worst_chunk0, worst = worst, 0.0
    if friction:
        print(f"   (chunk 1, start from rest: worst {worst_chunk0:.2e} against a calibrated bound of {max(bound[0].values()):.1e})")
    print(f"randomized assembly seed {seed} friction {friction}: n_arm {n_arm} n_elem {n_elem} dt {dt:.2e} worst {worst:.2e} "
          f"(worst err/bound {worst_ratio:.2f}; largest bound {max(max(b.values()) for b in bound):.1e})")
    h.close()


# ---- an env's bits depend on nothing but the env (VERDICT r1 item 4) ----------------------------------------------------
def _pendulum_batch(n_env, wild, steps, use_async):
    """SoftPendulum handle of n_env envs: env 0 is the probe (seed 42), the others are either well behaved or spin so
    fast that every one of them leaves the fast-math range at every step (they are re-run by the safe kernel, and after
    the first poll of the fallback counter the whole handle drops to the safe kernel alone).  Returns env 0's state after
    each step, the launch count per step, and the final count."""
    import torch
    from gym_softrobot_b200.envs.soft_pendulum import pendulum_init_params
    nat = _native()
    h = make_pendulum_handle(n_env, nat.MATH_FAST)
    u = np.array([u01_for_seed(42)] + [u01_for_seed(100 + i) for i in range(1, n_env)])
    h.reset_host(pendulum_init_params(u))
    if wild and n_env > 1:
        h.fields()["omega_collection"][1:, 2, 1:] = 3000.0     # 0.3 rad per substep about d3: out of the rotation range
    rng = np.random.default_rng(7)
    acts = rng.uniform(-22, 22, size=(steps, 1)).astype(np.float32)
    obs = torch.empty((n_env, 4), dtype=torch.float32, device="cuda")
    rew = torch.empty(n_env, dtype=torch.float64, device="cuda")
    term = torch.empty(n_env, dtype=torch.uint8, device="cuda")
    states, launches = [], []
    for s in range(steps):
        a = np.repeat(acts[s][None, :], n_env, axis=0)
        if use_async:
            h.step(torch.as_tensor(a, device="cuda"), 400, obs, rew, term)
            if s % 3 == 0:
                time.sleep(0.002 * (s % 5))       # perturb the host timing the adaptive switch could be sensitive to
        else:
            h.step_host(a, 400)
        states.append(h.state_tensor()[0].clone())
        launches.append(h.launch_count)
    torch.cuda.synchronize()
    h.close()
    return states, np.diff([1] + launches)


def test_env_bits_are_independent_of_the_batch_and_of_the_kernel_pair():
    """DESIGN.md §5 "bit-identical whatever the batch": one SoftPendulum env stepped 20 times (8000 substeps, actions
    from a fixed list) alone, among 15 well-behaved envs, and among 15 envs that all fall back — the last case crosses
    the handle-wide switch from the fast-only / fallback pair to the safe kernel alone (checked through the launch
    count), so it also shows that both kernels compute the same bits.  torch.equal on the whole state block, every step."""
    import torch
    alone, l_alone = _pendulum_batch(1, False, 20, False)
    calm, l_calm = _pendulum_batch(16, False, 20, False)
    wild, l_wild = _pendulum_batch(16, True, 20, False)
    assert np.all(l_alone == 2) and np.all(l_calm == 2)       # fast-only + (empty) fallback every step
    assert l_wild[0] == 2 and l_wild[-1] == 1, l_wild          # the pair switched itself off on the way
    for s in range(20):
        assert torch.equal(alone[s], calm[s]), f"step {s}: env 0 differs between a batch of 1 and a batch of 16"
        assert torch.equal(alone[s], wild[s]), f"step {s}: env 0 differs when its neighbours fall back / after the switch"
    assert torch.isfinite(alone[-1][:18]).all()


def test_async_path_is_reproducible_across_runs_and_host_timing():
    """Two runs of the stream-ordered sr_step path (device pointers, no host synchronisation) with different host-side
    timing, on a handle that crosses the adaptive switch: identical bits for the probe env, step by step."""
    import torch
    a, la = _pendulum_batch(16, True, 20, True)
    b, lb = _pendulum_batch(16, True, 20, False)
    c, lc = _pendulum_batch(16, True, 20, True)
    for s in range(20):
        assert torch.equal(a[s], b[s]) and torch.equal(a[s], c[s]), f"step {s}"


def test_contact_env_bits_are_independent_of_its_neighbours():
    """Same property for a generic-kernel instantiation (plane contact + rest curvature, OctoArmSingle's model): the
    probe arm's state is bit-identical alone, among calm arms, and among arms bent far outside the fast bend range."""
    import torch
    from gym_softrobot_b200.envs.arm_single import arm_contact_params, _ROD, _G
    nat = _native()

    def run(n_env, wild):
        h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=50, dt=7e-5, gravity=(0.0, 0.0, _G), damping_constant=1e-2,
                       bc_kind=nat.BC_FREE, contact=arm_contact_params(), **_ROD)
        init = np.zeros((n_env, 9)); init[:, 3] = 1.0; init[:, 8] = 1.0
        h.reset_host(init)
        s = np.linspace(0, 1, 49)
        rk = h.rest_kappa_tensor()
        rk[:, 0, :] = torch.as_tensor(8.0 * np.sin(np.pi * s), device="cuda")
        if wild and n_env > 1:
            rk[1:, 0, :] = 150.0      # ~60 degrees per element once relaxed: far outside the 37-degree map
        out = []
        for _ in range(12):
            h.step_host(None, 200)
            out.append(h.state_tensor()[0].clone())
        h.close()
        return out

    alone, calm, wild = run(1, False), run(11, False), run(11, True)
    for s in range(12):
        assert torch.equal(alone[s], calm[s]) and torch.equal(alone[s], wild[s]), f"step {s}"


# ---- groundwork for the muscle-driven octopus envs (VERDICT r1 item 8): tapered rods, sucker constraint, external loads ----
@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_tapered_rod_with_sucker_and_external_loads_vs_c_oracle(seed):
    """A single tapered arm (base_radius = linspace(base, tip, n): build_muscle_octopus.py:61-63), one end free or
    clamped, with a ControllableFixConstraint on node / element 0 (controllable_constraint.py:46-69), smooth external
    nodal forces (lab frame) and element couples (material frame) applied every substep as a forcing, gravity and the
    analytical damper; odd seeds add the frictionless plane.  CUDA (per-element constants from the HBM table) vs the
    C oracle (whose arrays are per element anyway), every field, 600 substeps, 1e-9."""
    import torch
    import rod_oracle as ro
    nat = _native()
    rng = np.random.default_rng(300 + seed)
    n = int(rng.choice([12, 25, 40, 63]))
    L, r_base = 0.2, 0.012
    r_tip = float(r_base * rng.uniform(0.08, 0.5))
    E, rho = 1e5, 1050.0
    dt = float(0.05 * (L / n) / np.sqrt(E / rho))
    bc = int(rng.choice([0, 1]))
    ratio = float(rng.uniform(0.0, 1.0))
    plane = dict(plane_origin=(0.0, 0.0, -r_base), plane_normal=(0.0, 0.0, 1.0), k=1e2, nu=1e1, slip_velocity_tol=1e-8,
                 static_mu=(0.0, 0.0, 0.0), kinetic_mu=(0.0, 0.0, 0.0)) if seed % 2 else None
    s_n, s_e = np.linspace(0, 1, n + 1), np.linspace(0, 1, n)
    # loads scaled with the local cross-section (a muscle's force goes with its area, its couple with area x radius)
    tn, te = (1 + (r_tip / r_base - 1) * s_n) ** 2, (1 + (r_tip / r_base - 1) * s_e) ** 3
    fext = 2e-3 * tn * np.stack([rng.uniform(-1, 1) * np.sin(np.pi * s_n), rng.uniform(-1, 1) * s_n, rng.uniform(-1, 1) * np.cos(np.pi * s_n)])
    cext = 2e-4 * te * np.stack([rng.uniform(-1, 1) * np.sin(np.pi * s_e), rng.uniform(-1, 1) * np.sin(2 * np.pi * s_e), rng.uniform(-1, 1) * s_e])
    o = ro.OracleRod(n, [0, 0, 0], [1.0, 0, 0], [0, 0, 1.0], L, r_base, rho, E, dt, gravity=(0.0, 0.0, -9.81),
                     damping_constant=0.05, bc_kind=bc, contact=plane, tip_radius=r_tip)
    o.user_forces[...] = fext; o.user_torques[...] = cext
    o.set_sucker(0, 0, ratio)
    n_env = 3
    h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n, dt=dt, base_length=L, base_radius=r_base, density=rho,
                   youngs_modulus=E, gravity=(0.0, 0.0, -9.81), damping_constant=0.05, bc_kind=bc, contact=plane,
                   tip_radius=r_tip, sucker_index=0)
    init = np.zeros((n_env, 9)); init[:, 3] = 1.0; init[:, 8] = 1.0
    h.reset_host(init)
    h.sucker_tensor()[:] = ratio
    f_t, c_t = h.ext_load_tensors()
    f_t[:] = torch.as_tensor(fext, device="cuda"); c_t[:] = torch.as_tensor(cext, device="cuda")
    worst = 0.0
    for chunk in (250, 350):
        h.step_host(None, chunk); o.substeps(chunk)
        f = {k: v.cpu().numpy() for k, v in h.fields().items()}
        for fk in FIELDS.values():
            ref = getattr(o, fk)
            err = float(np.abs(f[fk][1] - ref).max() / max(np.abs(ref).max(), ASM_FLOOR[fk] * 0.1))
            worst = max(worst, err)
            assert err < TOL, f"seed {seed} (n {n}, tip/base {r_tip / r_base:.2f}, bc {bc}, plane {plane is not None}) {fk}: {err:.3e}"
    assert np.abs(o.velocity_collection).max() > 1e-3      # the loads did move the arm
    print(f"tapered rod seed {seed}: n {n} tip/base {r_tip / r_base:.2f} bc {bc} plane {plane is not None} worst {worst:.2e}")
    h.close(); o.close()


def test_tapered_muscle_octopus_topology_vs_c_oracle():
    """The systems build_octopus_muscles assembles (build_muscle_octopus.py:70-179), minus the COOMM forcing: eight
    tapered arms at 22.5 + 45 i degrees around a light rigid head, FixedJoint2Rigid (kt = 1e2), dampers, no gravity,
    no plane; a sucker on node 0 of every arm (crawl_env.py:146-157) with per-arm ratios, and synthetic per-element
    external couples standing in for ApplyMuscles.  CUDA vs the multi-rod C oracle, every field, 600 substeps, 1e-9.

    Conditioning, measured here on the oracle itself: the reference's head is light (head_density 50, I ~ 3e-7 kg m^2)
    and held by kt = 1e2, so d(omega_head)/d(director) ~ kt dt / I ~ 3e3 per substep.  An oracle replica started 1e-13
    (relative) away in its arm positions ends 8e-12 .. 1.5e-11 away in head omega (3e-9 of |omega| = 2.7e-3): the 1e-9
    bar on that one field would need the whole state to 3e-14.  The check is therefore max(1e-9 scale, 20 x the
    replica's divergence) per field — the CUDA path has to stay as close to the oracle as an oracle started 2e-12 away;
    the one-ulp replica and the FMA-contracted build of the oracle are printed beside it for scale."""
    import torch
    import rod_oracle as ro
    nat = _native()
    rng = np.random.default_rng(77)
    n_arm, n, L, r_base, r_tip, head_radius = 8, 20, 0.2, 0.012, 0.0012, 0.02
    E, rho, dt = 1e5, 1050.0, 1e-5
    k, kt, nu, head_density = 1e4, 1e2, 1e-3, 50.0
    asm = ro.octopus_assembly(n_arm=n_arm, n_elem=n, time_step=dt, head_radius=head_radius, head_density=head_density,
                              body_arm_k=k, body_arm_kt=kt, body_arm_nu=nu, base_length=L, base_radius=r_base,
                              youngs_modulus=E, density=rho, tip_radius=r_tip, plane=False, gravity=0.0,
                              damping_constant=0.05, angle_offset=22.5)
    s_e = np.linspace(0, 1, n)
    ratios = rng.uniform(0, 1, n_arm)
    te = (1 + (r_tip / r_base - 1) * s_e) ** 3
    cext = np.stack([2e-4 * te * np.stack([rng.uniform(-1, 1) * np.sin(np.pi * s_e), rng.uniform(-1, 1) * np.sin(np.pi * s_e),
                                            0.2 * rng.uniform(-1, 1) * s_e]) for _ in range(n_arm)])
    for a, rod in enumerate(asm.arms):
        rod.user_torques[...] = cext[a]
        rod.set_sucker(0, 0, ratios[a])
    n_env = 2
    angles = [22.5 + 45.0 * a for a in range(n_arm)]
    h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n, dt=dt, base_length=L, base_radius=r_base, density=rho,
                   youngs_modulus=E, gravity=(0.0, 0.0, 0.0), damping_constant=0.05, bc_kind=nat.BC_FREE, n_rod=n_arm,
                   head=dict(length=2 * r_base, radius=head_radius, density=head_density),
                   joint=dict(radius=head_radius, angles_deg=angles, k=k, nu=nu, kt=kt), tip_radius=r_tip, sucker_index=0)
    row = []
    for ang in angles:
        c, s = np.cos(np.deg2rad(ang)), np.sin(np.deg2rad(ang))
        row += [c * head_radius, s * head_radius, 0.0, c, s, 0.0, 0.0, 0.0, 1.0]
    row += [0.0, 0.0, -r_base, 0.0, 0.0, 1.0, 0.0, 1.0, 0.0]
    h.reset(torch.as_tensor(np.repeat(np.array([row]), n_env, axis=0), device="cuda").contiguous())
    h.sucker_tensor().unflatten(0, (n_env, n_arm))[:] = torch.as_tensor(ratios, device="cuda")
    f_t, c_t = h.ext_load_tensors()
    c_t.unflatten(0, (n_env, n_arm))[:] = torch.as_tensor(cext, device="cuda")
    o6 = torch.empty((n_env, 6), dtype=torch.float32, device="cuda")
    rew = torch.empty(n_env, dtype=torch.float64, device="cuda")
    term = torch.empty(n_env, dtype=torch.uint8, device="cuda")
    # the oracle's own one-ulp sensitivity (arms that have barely started to move amplify position round-off through
    # the stiff joint springs): a replica whose arm positions sit on neighbouring doubles
    def make():
        a2 = ro.octopus_assembly(n_arm=n_arm, n_elem=n, time_step=dt, head_radius=head_radius, head_density=head_density,
                                 body_arm_k=k, body_arm_kt=kt, body_arm_nu=nu, base_length=L, base_radius=r_base,
                                 youngs_modulus=E, density=rho, tip_radius=r_tip, plane=False, gravity=0.0,
                                 damping_constant=0.05, angle_offset=22.5)
        for a, rod in enumerate(a2.arms):
            rod.user_torques[...] = cext[a]
            rod.set_sucker(0, 0, ratios[a])
        return a2
    rep = make()
    prng = np.random.default_rng(5)
    for rod in rep.arms:
        x = rod.position_collection
        x[...] = np.nextafter(x, np.where(prng.random(x.shape) < 0.5, -np.inf, np.inf))
    # ... the same C source built with FMA contraction (oracle/Makefile): two correct builds of ONE implementation
    with ro.variant("fma"):
        rep_fma = make()
    # ... and the replica 1e-13 away (docstring)
    rep_13 = make()
    for rod in rep_13.arms:
        rod.position_collection[...] *= 1.0 + 1e-13 * prng.standard_normal(rod.position_collection.shape)
    reps = (rep, rep_fma, rep_13)
    head_sens = {}
    worst, worst_rel = 0.0, 0.0
    for chunk in (300, 300):
        h.step(None, chunk, o6, rew, term); asm.substeps(chunk)
        for r_ in reps:
            r_.substeps(chunk)
        f = {k_: v.cpu().numpy() for k_, v in h.fields().items()}
        hd = h.head_tensor().cpu().numpy()
        assert int(term.sum()) == 0
        for a, rod in enumerate(asm.arms):
            for fk in FIELDS.values():
                ref = getattr(rod, fk)
                sens = max(float(np.abs(getattr(r_.arms[a], fk) - ref).max()) for r_ in reps)
                err_abs = float(np.abs(f[fk][1, a] - ref).max())
                scale = max(float(np.abs(ref).max()), ASM_FLOOR[fk])
                worst, worst_rel = max(worst, err_abs / scale), max(worst_rel, err_abs / max(TOL * scale, 20 * sens))
                assert err_abs < max(TOL * scale, 20 * sens), f"arm {a} {fk}: {err_abs / scale:.3e} (one-ulp divergence of the oracle {sens / scale:.1e})"
        mine = np.concatenate([asm.head_position, asm.head_velocity, asm.head_director.reshape(-1), asm.head_omega])
        repl = [np.concatenate([r_.head_position, r_.head_velocity, r_.head_director.reshape(-1), r_.head_omega])
                for r_ in reps]
        for sl, fk in HEAD_SLICES:
            scale = max(float(np.abs(mine[sl]).max()), ASM_FLOOR[fk])
            err_abs, sens = float(np.abs(hd[1, sl] - mine[sl]).max()), max(float(np.abs(r_[sl] - mine[sl]).max()) for r_ in repl)
            worst = max(worst, err_abs / scale)
            head_sens[fk] = [float(np.abs(r_[sl] - mine[sl]).max()) / scale for r_ in repl] + [err_abs / scale]
            assert err_abs < max(TOL * scale, 20 * sens), f"head {fk}: {err_abs / scale:.3e} (replicas one-ulp / fma / 1e-13: {head_sens[fk][:3]})"
    for r_ in reps:
        r_.close()
    print(f"tapered muscle-octopus topology: worst {worst:.2e}; head omega [one-ulp, fma build, 1e-13 replica, CUDA] = "
          + ", ".join(f"{v:.1e}" for v in head_sens["omega_collection"]))
    h.close(); asm.close()


def test_two_handles_on_two_devices_agree():
    """The opt-in above 48 KB of dynamic shared memory is a per-device attribute of a kernel (cudaFuncSetAttribute):
    a second handle on another device of the same process has to set it again (round-1 advisory).  Two SoftPendulum
    handles (lean kernel, split schedule: 600 envs > resident slots) and two contact handles (lean plane model) on
    cuda:0 and cuda:1 are stepped through host buffers, interleaved, and must agree bit for bit."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs (gpurun --gpus 2)")
    from gym_softrobot_b200.envs.soft_pendulum import _make_handle, pendulum_init_params
    from gym_softrobot_b200.envs.arm_single import arm_contact_params, _ROD, _G
    nat = _native()
    n_env = 600
    hs = [_make_handle(n_env, 50, 1e-4, d, nat.MATH_FAST) for d in (0, 1)]
    u = np.array([u01_for_seed(42 + i) for i in range(n_env)])
    acts = np.random.default_rng(3).uniform(-22, 22, size=(3, n_env, 1)).astype(np.float32)
    for h in hs:
        h.reset_host(pendulum_init_params(u))
    outs = []
    for s in range(3):
        outs.append([h.step_host(acts[s], 400) for h in hs])
    for s in range(3):
        for a, b in zip(outs[s][0], outs[s][1]):
            assert np.array_equal(np.asarray(a), np.asarray(b)), f"SoftPendulum step {s}: devices disagree"
    st = [h.fields()["velocity_collection"].cpu().numpy() for h in hs]
    assert np.array_equal(st[0], st[1]) and np.isfinite(st[0]).all()
    for h in hs:
        h.close()
    cs = [nat.Handle(model=nat.MODEL_ROD, n_env=64, n_elem=50, dt=7e-5, gravity=(0.0, 0.0, _G), damping_constant=1e-2,
                     bc_kind=nat.BC_FREE, contact=arm_contact_params(), device=d, **_ROD) for d in (1, 0)]
    init = np.zeros((64, 9)); init[:, 3] = 1.0; init[:, 8] = 1.0
    for h in cs:
        h.reset_host(init)
        h.rest_kappa_tensor()[:, 0, :] = torch.as_tensor(np.linspace(-4, 4, 64)[:, None] * np.ones((1, 49)), device=f"cuda:{h.device}")
        h.step_host(None, 300)
    st = [h.fields()["position_collection"].cpu().numpy() for h in cs]
    assert np.array_equal(st[0], st[1]) and np.isfinite(st[0]).all()
    for h in cs:
        h.close()


def test_split_schedule_keeps_every_lean_variant_bit_identical():
    """The lean kernel deals work by substep count: with more env groups than resident CTA slots an item is started by
    one CTA and finished by another, its registers (and the travelling wave's phase, the assembly's head, the moving
    base's command) travelling through global scratch.  For every variant — plain, contact, contact + muscle wave,
    assembly, filter + moving base, spline torques — a batch of IDENTICAL envs large enough to be split must come out
    identical in every env, wherever the schedule cut the env's item, and equal to a batch small enough not to be split.
    (This is the test that caught the moving base being reset to its finalize-time anchor on resume.)"""
    import torch
    import gym_softrobot_b200 as g
    from gym_softrobot_b200.envs.arm_single import arm_contact_params, _ROD, _G
    from gym_softrobot_b200.envs.octo_flat import OctoFlatVectorEnv
    from gym_softrobot_b200.envs.soft_pendulum import pendulum_init_params
    nat = _native()
    sm = torch.cuda.get_device_properties(0).multi_processor_count

    def same_everywhere(t, group, name):
        ref = t[:group]
        n = t.shape[0] // group
        eq = (t.reshape(n, group, *t.shape[1:]) == ref[None]).flatten(1).all(dim=1)
        assert bool(eq.all()), f"{name}: {int((~eq).sum())} of {n} identical envs differ from env 0 (first: {int((~eq).nonzero()[0])})"
        return ref.clone()

    def plain(n_env, dtype=None):
        from gym_softrobot_b200.envs.soft_pendulum import _make_handle
        h = make_pendulum_handle(n_env, nat.MATH_FAST) if dtype is None else _make_handle(n_env, 50, 1e-4, 0, nat.MATH_FAST, dtype)
        h.reset_host(pendulum_init_params(np.full(n_env, u01_for_seed(42))))
        a = np.full((n_env, 1), 7.5, dtype=np.float32)
        for _ in range(3):
            h.step_host(a, 333)
        out = same_everywhere(h.state_tensor(), 1, "plain" if dtype is None else "plain, FP32 storage")
        h.close()
        return out

    def plain_f32(n_env):
        return plain(n_env, nat.DTYPE_F32)

    def contact(n_env):
        h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=50, dt=7e-5, gravity=(0.0, 0.0, _G), damping_constant=1e-2,
                       bc_kind=nat.BC_FREE, contact=arm_contact_params(), **_ROD)
        init = np.zeros((n_env, 9)); init[:, 3] = 1.0; init[:, 8] = 1.0
        h.reset_host(init)
        h.rest_kappa_tensor()[:, 0, :] = torch.as_tensor(8.0 * np.sin(np.pi * np.linspace(0, 1, 49)), device="cuda")
        for _ in range(3):
            h.step_host(None, 333)
        out = same_everywhere(h.state_tensor(), 1, "contact")
        h.close()
        return out

    def fold(n_env):     # 512 elements: one rod per CTA, the tip node folded into the last thread and handed over with it
        h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=512, dt=5e-6, gravity=(0.0, 0.0, _G), damping_constant=1e-2,
                       bc_kind=nat.BC_FREE, contact={**arm_contact_params(), "plane_origin": [0.0, 0.0, -0.005]}, base_length=1.0,
                       base_radius=0.005, density=1000.0, youngs_modulus=1e6)
        init = np.zeros((n_env, 9)); init[:, 3] = 1.0; init[:, 8] = 1.0
        h.reset_host(init)
        h.rest_kappa_tensor()[:, 0, :] = torch.as_tensor(3.0 * np.sin(np.linspace(0, 3 * np.pi, 511)), device="cuda")
        for _ in range(3):
            h.step_host(None, 133)
        out = same_everywhere(h.state_tensor(), 1, "folded tip")
        h.close()
        return out

    def snake(n_env):
        env = g.make_vec("ContinuumSnake-v0", n_env, autoreset=False); env.reset()
        mu = env.handle.muscle_tensor()
        mu[:, 2:] = torch.as_tensor(np.random.default_rng(3).uniform(-4e-3, 4e-3, (1, 6)), device="cuda") @ env._W.T
        mu[:, 1] = 2 * np.pi / 0.97
        o6, rew, term = env._scratch
        for _ in range(3):
            env.handle.step(None, 333, o6, rew, term)
        out = (same_everywhere(env.handle.state_tensor(), 1, "snake"), same_everywhere(mu, 1, "snake clock"))
        env.close()
        return out

    def assembly(n_env):
        env = OctoFlatVectorEnv(n_env, n_elems=10, time_step=7e-5, autoreset=False); env.reset(seed=42)
        env.handle.rest_kappa_tensor()[:, 0, :] = torch.as_tensor(np.linspace(-5, 5, 8)[:, None] * np.ones((1, 9)), device="cuda").repeat(n_env, 1)
        o6, rew, term = env._scratch
        for _ in range(3):
            env.handle.step(None, 333, o6, rew, term)
        out = (same_everywhere(env.handle.state_tensor(), 8, "assembly arms"), same_everywhere(env.handle.head_tensor(), 1, "assembly head"))
        env.close()
        return out

    def filt(n_env):
        from gym_softrobot_b200.envs.soft_pendulum_3d import pendulum3d_init_params
        env = g.make_vec("SoftPendulum3D-v0", n_env, autoreset=False); env.reset(seed=42)
        env.handle.reset(torch.as_tensor(pendulum3d_init_params(np.full(n_env, 0.37)), device="cuda").contiguous())   # every env alike
        a = torch.as_tensor(np.tile(np.array([[1.0, -0.8]], dtype=np.float32), (n_env, 1)), device="cuda")
        for _ in range(12):           # the base walks 12 mm away from its finalize-time anchor (element length 20 mm)
            env.handle.step(a, 200, env.obs, env.reward, env.terminated)
        out = (same_everywhere(env.handle.state_tensor(), 1, "filter"), same_everywhere(env.handle.aux_tensor(), 1, "filter base"),
               same_everywhere(env.obs, 1, "filter obs"))
        assert env.handle.fallback_count() == 0, env.handle.fallback_causes()
        env.close()
        return out

    def spline(n_env):
        env = g.make_vec("SoftArmTracking-v0", n_env, autoreset=False); env.reset(seed=1)   # (the arm's build has no randomness)
        pts, mags = env.handle.spline_tensors()
        o6 = torch.empty((n_env, 6), dtype=torch.float32, device="cuda"); rew = torch.empty(n_env, dtype=torch.float64, device="cuda")
        term = torch.empty(n_env, dtype=torch.uint8, device="cuda")
        for k in range(3):
            pts[:, :, :env.handle.cfg.spline_n_ctrl] = 0.3 - 0.25 * k
            env.handle.step(None, 333, o6, rew, term)
        out = (same_everywhere(env.handle.state_tensor(), 1, "spline"), same_everywhere(mags, 1, "spline cache"))
        env.close()
        return out

    # (envs per CTA: 10 / 12 single rods in 512 threads, 4 assemblies of 89 threads in 384; a split needs more items than SMs)
    for name, fn, small, big in (("plain", plain, 20, 10 * sm + 1500), ("plain-f32", plain_f32, 20, 10 * sm + 1500),
                                 ("contact", contact, 20, 10 * sm + 1500), ("fold", fold, 3, sm + 61),
                                 ("snake", snake, 20, 10 * sm + 1500), ("assembly", assembly, 8, 4 * sm + 300),
                                 ("filter", filt, 20, 10 * sm + 1500), ("spline", spline, 24, 12 * sm + 1500)):
        a, b = fn(small), fn(big)
        a, b = (a, b) if isinstance(a, tuple) else ((a,), (b,))
        for ta, tb in zip(a, b):
            assert torch.equal(ta, tb), f"{name}: split and unsplit batches differ"
            assert torch.isfinite(tb).all(), name


@pytest.mark.parametrize("normal", [(0.3, -0.2, 1.0), (0.0, -1.0, 0.0), (0.0, 0.0, -1.0)], ids=["oblique", "minus-y", "minus-z"])
def test_rod_on_a_tilted_frictional_plane_vs_c_oracle(normal):
    """The contact kernels work in a frame whose z axis is the plane normal and rotate lab vectors on load / store; the
    reference envs only ever use +z (octopus) and +y (snake).  Here the plane is tilted (a genuinely non-permutation
    rotation), or flipped: an actuated rod lying on it under a gravity that presses it onto the plane and drags it
    sideways, sliding from the start (kinetic regime).  CUDA vs the C oracle (which takes dot products with the normal as
    PyElastica does), every field, 600 substeps, 1e-9."""
    import torch
    import rod_oracle as ro
    from gym_softrobot_b200.envs.arm_single import curvature_interp_matrix, _ROD
    nat = _native()
    N = np.array(normal, dtype=float); N /= np.linalg.norm(N)
    a = np.cross(N, [1.0, 0.0, 0.0]); a /= np.linalg.norm(a)        # rod axis, in the plane
    b = np.cross(N, a)                                               # second in-plane direction
    n_env, n, dt = 4, 50, 7e-5
    r0 = _ROD["base_radius"]
    c = _arm_contact(False)
    c["plane_origin"] = list(-r0 * N); c["plane_normal"] = list(N)
    grav = tuple(-9.81 * N + 1.5 * b)
    h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n, dt=dt, gravity=grav, damping_constant=1e-2,
                   bc_kind=nat.BC_FREE, contact=c, **_ROD)
    init = np.zeros((n_env, 9)); init[:, 3:6] = a; init[:, 6:9] = N
    h.reset_host(init)
    W = curvature_interp_matrix(7, n - 1)
    rk = np.random.default_rng(11).uniform(-8, 8, size=(n_env, 7)) @ W.T
    h.rest_kappa_tensor()[:, 0, :] = torch.as_tensor(rk, device="cuda")
    v0 = 0.05 * a + 0.03 * b
    h.fields()["velocity_collection"][:] = torch.as_tensor(v0, device="cuda")[None, :, None]
    rods = [ro.OracleRod(n, [0, 0, 0], list(a), list(N), _ROD["base_length"], r0, 1000.0, 1e6, dt,
                         gravity=grav, damping_constant=1e-2, contact=c) for _ in range(n_env)]
    for i, r in enumerate(rods):
        r.rest_kappa[0, :] = rk[i]
        r.velocity_collection[...] = v0[:, None]
    for chunk in (300, 300):
        h.step_host(None, chunk)
        f = {k: v.cpu().numpy() for k, v in h.fields().items()}
        for i, r in enumerate(rods):
            r.substeps(chunk)
            for name in ("position_collection", "velocity_collection", "director_collection", "omega_collection", "kappa", "tangents"):
                assert_state_close(f[name][i], getattr(r, name), name, {}, f"env {i}", TOL)
    # it slid along the plane and stayed on it
    x = f["position_collection"][0]
    height = (N[:, None] * x).sum(0)
    assert np.abs(height).max() < 5e-3 and np.abs((b[:, None] * x).sum(0)).max() > 1e-4
    h.close()


@pytest.mark.parametrize("seed", range(6))
def test_randomized_contact_rods_vs_c_oracle(seed):
    """The lean kernel's plane model over its whole configuration space, drawn per seed: rod size (12..160 elements:
    different CTA shapes and rods per CTA), material, plane orientation (arbitrary normal), free or clamped base, rest
    curvature about both bending axes and twist, friction coefficients, slip tolerance, contact spring and damping, the
    order of contact vs forcing, gravity pressing the rod onto the plane at an angle, and an initial slide.  CUDA vs the C
    oracle, six fields, 2 x 200 substeps, 1e-9 (or 20 x the oracle's own one-ulp divergence, measured)."""
    import torch
    import rod_oracle as ro
    nat = _native()
    rng = np.random.default_rng(5000 + seed)
    n = int(rng.choice([12, 25, 50, 63, 100, 160]))
    L, r0 = float(rng.uniform(0.15, 0.4)), float(rng.uniform(0.006, 0.012))
    E, rho = float(10 ** rng.uniform(5.5, 6.5)), float(rng.uniform(800, 1500))
    dt = float(0.04 * (L / n) / np.sqrt(E / rho))
    N = rng.normal(size=3); N /= np.linalg.norm(N)
    a = np.cross(N, rng.normal(size=3)); a /= np.linalg.norm(a)
    b = np.cross(N, a)
    bc = [nat.BC_FREE, nat.BC_ONE_END_FIXED][seed % 2]
    c = dict(plane_origin=list(-r0 * N), plane_normal=list(N), k=float(10 ** rng.uniform(1.5, 2.5)), nu=float(10 ** rng.uniform(0, 1.2)),
             slip_velocity_tol=float(10 ** rng.uniform(-6, -3)), static_mu=list(rng.uniform(0.2, 1.0, 3)),
             kinetic_mu=list(rng.uniform(0.1, 0.6, 3)), before_forcing=bool(rng.integers(2)))
    grav = tuple(-9.81 * N + rng.uniform(-2, 2) * a + rng.uniform(-2, 2) * b)
    damping = float(10 ** rng.uniform(-3, -1.5))
    kw = dict(gravity=grav, damping_constant=damping, contact=c, bc_kind=bc)
    n_env = 3
    h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n, dt=dt, base_length=L, base_radius=r0, density=rho, youngs_modulus=E, **kw)
    init = np.zeros((n_env, 9)); init[:, 3:6] = a; init[:, 6:9] = N
    h.reset_host(init)
    s = np.linspace(0, 1, n - 1)
    rk = np.stack([rng.uniform(-6, 6) * np.sin(np.pi * s * rng.integers(1, 3)), rng.uniform(-6, 6) * np.cos(np.pi * s), rng.uniform(-2, 2) * s])
    h.rest_kappa_tensor()[:] = torch.as_tensor(rk, device="cuda")[None]
    v0 = rng.uniform(-0.1, 0.1) * a + rng.uniform(-0.1, 0.1) * b
    if bc == nat.BC_FREE:
        h.fields()["velocity_collection"][:] = torch.as_tensor(v0, device="cuda")[None, :, None]

    def make():
        r = ro.OracleRod(n, [0, 0, 0], list(a), list(N), L, r0, rho, E, dt, **kw)
        r.rest_kappa[...] = rk
        if bc == nat.BC_FREE:
            r.velocity_collection[...] = v0[:, None]
        return r
    names = ("position_collection", "velocity_collection", "director_collection", "omega_collection", "kappa", "tangents")
    o = make()
    done = 0
    for chunk in (200, 200):
        h.step_host(None, chunk); o.substeps(chunk); done += chunk
        assert np.isfinite(o.position_collection).all(), "unstable random case (test generator problem)"
        sens = one_ulp_divergence(make, lambda rod: rod.substeps(done), {k: getattr(o, k).copy() for k in names})
        f = {k: v.cpu().numpy() for k, v in h.fields().items()}
        floors = rate_floors(E, rho, L, n, r0, np.abs(o.position_collection).max())
        for name in names:
            assert_state_close(f[name][1], getattr(o, name), name, floors, f"seed={seed} n={n} bc={bc} substeps={done}", measured=sens)
    h.close(); o.close()


@pytest.mark.parametrize("n_elem,bc,damp_first", [(8, 1, False), (9, 0, True), (13, 1, True), (20, 0, False), (63, 1, False), (100, 1, True), (160, 0, False)])
def test_filtered_rods_vs_c_oracle(n_elem, bc, damp_first):
    """The LaplaceDissipationFilter (order 7) outside SoftPendulum3D-v0's one shape: rods of 8 (the filter model's minimum: one
    reflection per end) to 160 elements, free or clamped, both dampen / constrain orders, swinging under gravity from a
    tilted start.  The lean kernel evaluates passes 1..6 as one 13-tap stencil on ghost-padded records; the C oracle
    runs the reference's seven passes.  Every field, after 500 and 800 substeps, 1e-9 — or 20 x the oracle's own divergence, measured
    two ways (one-ulp start; FMA-contracted build).  (This test is what exposed the first-order treatment of the
    reference's 1e-14 rotation guard: clamped rods starting from rest showed 2e-9 in omega until the guard was made exact,
    scripts/diag_omega.py.)"""
    import rod_oracle as ro
    nat = _native()
    L, r0, E, rho = 1.0, 0.05, 1e6, 2000.0
    dt = float(0.03 * (L / n_elem) / np.sqrt(E / rho))
    ang = np.deg2rad(5.0)        # nearly horizontal: gravity swings it hard from the first substep
    d = np.array([np.cos(ang), 0.0, np.sin(ang)]); nn = np.array([0.0, 1.0, 0.0])
    kw = dict(gravity=(0.0, 0.0, -9.80665), damping_constant=0.3, laplace_filter_order=7, bc_kind=bc, damping_before_constraints=damp_first)
    n_env = 3
    h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n_elem, dt=dt, base_length=L, base_radius=r0, density=rho, youngs_modulus=E, **kw)
    init = np.zeros((n_env, 9)); init[:, 3:6] = d; init[:, 6:9] = nn
    h.reset_host(init)
    v0 = np.array([0.0, 0.3, 0.0])
    if bc == nat.BC_FREE:
        h.fields()["velocity_collection"][:] = __import__("torch").as_tensor(v0, device="cuda")[None, :, None]

    def make():
        o = ro.OracleRod(n_elem, [0, 0, 0], list(d), list(nn), L, r0, rho, E, dt, **kw)
        if bc == nat.BC_FREE:
            o.velocity_collection[...] = v0[:, None]
        return o
    names = ("position_collection", "velocity_collection", "director_collection", "omega_collection", "kappa", "sigma")
    o = make()
    done = 0
    for chunk in (500, 300):
        h.step_host(None, chunk); o.substeps(chunk); done += chunk
        ref = {k: getattr(o, k).copy() for k in names}
        s1, s2 = one_ulp_divergence(make, lambda rod: rod.substeps(done), ref), fma_build_divergence(make, lambda rod: rod.substeps(done), ref)
        sens = {k: max(s1[k], s2[k]) for k in names}
        f = {k: v.cpu().numpy() for k, v in h.fields().items()}
        floors = rate_floors(E, rho, L, n_elem, r0, np.abs(o.position_collection).max())
        for name in names:
            assert_state_close(f[name][1], getattr(o, name), name, floors, f"n={n_elem} bc={bc} substeps={done}", measured=sens)
    assert h.fallback_count() == 0
    h.close(); o.close()
