"""Device-timed throughput of the non-headline kernel instantiations (contact, SoftPendulum3D, assemblies, long rod):
one JSON line each.  A/B switches come from the environment (SOFTROD_FASTPATH, SOFTROD_LEAN_FOLD, ...: INTEGRATION.md §6)
and are recorded in each line."""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
import gym_softrobot_b200 as g
from gym_softrobot_b200 import _native as nat
from gym_softrobot_b200.envs.arm_single import arm_contact_params, _ROD
which = sys.argv[1].split(",") if len(sys.argv) > 1 else ["contact50", "sp3d", "multi10", "multi40", "contact512", "snake", "softarm"]
peak = nat.measure_fp64_peak(0)

def timed(fn, K=6, W=3):
    for _ in range(W): fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for a, b in ev:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    return sorted(a.elapsed_time(b) for a, b in ev)[K // 2] * 1e-3

def report(name, n_env, elems, K, sec, flop, handle=None):
    es = n_env * elems * K / sec
    print(json.dumps(dict(config=name, fallback_env_steps=(handle.fallback_count() if handle is not None else None), launches=(handle.launch_count if handle is not None else None), n_env=n_env, ms_per_step=round(sec * 1e3, 4), elem_substeps_per_s=es, fp64_frac=round(es * flop / 1e12 / peak, 4),
                          knobs={k: v for k, v in os.environ.items() if k.startswith("SOFTROD_")})), flush=True)

def outs(n_env):
    return (torch.empty((n_env, 6), dtype=torch.float32, device="cuda"), torch.empty(n_env, dtype=torch.float64, device="cuda"),
            torch.empty(n_env, dtype=torch.uint8, device="cuda"))

if "contact50" in which:
    n_env = 4096
    h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=50, dt=7e-5, gravity=(0, 0, -9.81), damping_constant=1e-2,
                   bc_kind=nat.BC_FREE, contact=arm_contact_params(), **_ROD)
    init = np.zeros((n_env, 9)); init[:, 3] = 1.0; init[:, 8] = 1.0
    h.reset_host(init)
    h.rest_kappa_tensor()[:, 0, :] = torch.as_tensor(np.random.default_rng(1).uniform(-5, 5, (n_env, 1)) * np.ones((1, 49)), device="cuda")
    o, r, t = outs(n_env)
    report("rod on frictional plane n=50 (OctoArmSingle model)", n_env, 50, 400, timed(lambda: h.step(None, 400, o, r, t)), 720, h)
    assert int(t.sum()) == 0; h.close()
if "sp3d" in which:
    n_env = 4096
    env = g.make_vec("SoftPendulum3D-v0", n_env, autoreset=False); env.reset(seed=42)
    a = (torch.rand((n_env, 2), device="cuda") * 2 - 1).float()
    report("SoftPendulum3D-v0", n_env, 50, 400, timed(lambda: env.handle.step(a, 400, env.obs, env.reward, env.terminated)), 608, env.handle)
    env.close()
from gym_softrobot_b200.envs.octo_flat import OctoFlatVectorEnv
for tag, n_elem, n_env, dt in (("multi10", 10, 16384, 7e-5), ("multi40", 40, 4096, 3e-5)):
    if tag not in which: continue
    env = OctoFlatVectorEnv(n_env, n_elems=n_elem, time_step=dt, autoreset=False); env.reset(seed=42)
    env.handle.rest_kappa_tensor()[:, 0, :] = torch.as_tensor(np.random.default_rng(2).uniform(-5, 5, (n_env * 8, 1)) * np.ones((1, n_elem - 1)), device="cuda")
    o6, rew, term = env._scratch
    report(f"8-arm assembly n_elem={n_elem}", n_env, 8 * n_elem, 400, timed(lambda: env.handle.step(None, 400, o6, rew, term), K=4), 720, env.handle)
    assert int(term.sum()) == 0; env.close()
if "contact512" in which:
    n_env = 4096
    h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=512, dt=5e-6, gravity=(0, 0, -9.81), damping_constant=1e-2, bc_kind=nat.BC_FREE,
                   contact={**arm_contact_params(), "plane_origin": [0.0, 0.0, -0.005]}, base_length=1.0, base_radius=0.005, density=1000.0, youngs_modulus=1e6)
    init = np.zeros((n_env, 9)); init[:, 3] = 1.0; init[:, 8] = 1.0
    h.reset_host(init)
    h.rest_kappa_tensor()[:, 0, :] = torch.as_tensor(np.random.default_rng(1).uniform(-3, 3, (n_env, 1)) * np.ones((1, 511)), device="cuda")
    o, r, t = outs(n_env)
    report("long slender rod n=512 on frictional plane", n_env, 512, 50, timed(lambda: h.step(None, 50, o, r, t)), 720, h)
    assert int(t.sum()) == 0; h.close()
if "snake" in which:
    n_env = 4096
    env = g.make_vec("ContinuumSnake-v0", n_env, autoreset=False); env.reset()
    mu = env.handle.muscle_tensor()
    mu[:, 2:] = torch.as_tensor(np.random.default_rng(3).uniform(-4e-3, 4e-3, (n_env, 6)), device="cuda") @ env._W.T
    mu[:, 1] = 2 * np.pi / 0.97
    o6, rew, term = env._scratch
    report("ContinuumSnake-v0 (400-substep segment)", n_env, 50, 400, timed(lambda: env.handle.step(None, 400, o6, rew, term), K=4), 840, env.handle)
    env.close()
if "softarm" in which:
    n_env = 16384
    env = g.make_vec("SoftArmTracking-v0", n_env, autoreset=False); env.reset(seed=1)
    o6, rew, term = outs(n_env)
    pts, mags = env.handle.spline_tensors()
    pts[:, :, :env.handle.cfg.spline_n_ctrl] = 0.3
    report("SoftArmTracking-v0 kernel (400 substeps)", n_env, 40, 400, timed(lambda: env.handle.step(None, 400, o6, rew, term), K=4), 460, env.handle)
    env.close()
