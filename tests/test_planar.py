"""The planar model of the lean kernel (rod_kernel_lean.cuh): rods that stay in the lab x-y plane are stepped
with the out-of-plane terms left out, and must give the bits of the 3D kernels (DESIGN.md §5).

CPU: the C oracle keeps every out-of-plane component exactly zero, for SoftPendulum-v0 and for every clamped, free and
slider rod the host hands to the planar kernel (the premise of the model); the shape table below follows the host's
CTA rule.
GPU: each case runs in a subprocess per kernel setting — SOFTROD_LEAN_PLANAR=0 (3D kernels), the default (planar) and,
for the range fallbacks, SOFTROD_FASTPATH=0 (safe kernel only) — and the whole state block, observations, rewards and
termination flags must be equal.  The planar rods are also compared with the C oracle."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BC_FREE, BC_ONE_END_FIXED, BC_PENDULUM_SLIDER = 0, 1, 2     # (= _native / rod_oracle)

# n_elem -> (CTA threads, rods per CTA, barriers) of the lean kernel (lean_threads_setting, softrod_api.cu; per-rod
# named barriers need >= 32 threads per rod and 2..15 rods per CTA, rod_kernel_lean.cuh).  3: 128 rods per CTA; 31 / 32:
# either side of the named-barrier boundary, 32 with warps shared by two rods; 256: one rod per CTA with CTA-wide
# barriers; 383 / 511: full CTAs; 384: 127 idle threads.
SHAPES = {3: (512, 128, "cta"), 7: (512, 64, "cta"), 31: (512, 16, "cta"), 32: (512, 15, "named"),
          50: (512, 10, "named"), 95: (384, 4, "named"), 191: (384, 2, "named"), 255: (512, 2, "named"),
          256: (384, 1, "cta"), 383: (384, 1, "cta"), 384: (512, 1, "cta"), 511: (512, 1, "cta")}
PROBE = 1             # the env of every B batch that is tilted out of the plane
LAUNCHES = (400, 600)  # substeps of the two launches of every shape case


def test_oracle_keeps_soft_pendulum_in_its_plane():
    """x_z, v_z, d1_z, d3_z, d2_x, d2_y, w_0, w_2, kappa_0, kappa_2 and sigma_1 are exactly 0.0 over 2 x 8 env-steps of
    random +-22 actions (6400 substeps), while the in-plane motion is not small."""
    import rod_oracle as ro
    rng = np.random.default_rng(0)
    for seed in range(2):
        e = ro.OracleSoftPendulum()
        e.reset(seed=seed)
        r = e.rod
        for _ in range(8):
            e.step(np.float32(rng.uniform(-22, 22)))
            _assert_in_plane(r, seed)
        assert np.abs(r.omega_collection[1]).max() > 1e-3 and np.abs(r.velocity_collection[:2]).max() > 1e-3


def _out_of_plane(r):
    Q = r.director_collection
    return {"x_z": r.position_collection[2], "v_z": r.velocity_collection[2], "d1_z": Q[0, 2], "d3_z": Q[2, 2],
            "d2_xy": Q[1, :2], "w_0": r.omega_collection[0], "w_2": r.omega_collection[2], "kappa_02": r.kappa[[0, 2]],
            "sigma_1": r.sigma[1]}


def _assert_in_plane(r, what):
    for name, a in _out_of_plane(r).items():
        assert np.all(a == 0.0), (what, name, float(np.abs(a).max()))


_WORKER = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from gym_softrobot_b200 import _native as nat
from gym_softrobot_b200.envs.soft_pendulum import _make_handle, pendulum_init_params
case, out = sys.argv[2], sys.argv[3]
rng = np.random.default_rng(11)
if case in ("pendulum", "mixed"):
    n = 4096 if case == "pendulum" else 64
    h = _make_handle(n, 50, 1e-4, 0, nat.MATH_FAST)
    init = pendulum_init_params(rng.random(n))
    if case == "mixed":
        # env 5 is reset with its rod tilted 0.02 rad out of the plane (normal unchanged, still orthogonal)
        phi = 0.02
        init[5, 3] *= np.cos(phi); init[5, 4] *= np.cos(phi); init[5, 5] = np.sin(phi)
    h.reset_host(init)
    if case == "mixed":
        fl = h.fields()       # and two envs are pushed out of it through the state
        fl["omega_collection"][9, 0, 10] = 0.5
        fl["position_collection"][17, 2, 30] = 1e-4
        import torch
        torch.cuda.synchronize()     # (the handle steps on a stream of its own)
    steps, acts = (10 if case == "pendulum" else 12), True
else:
    # BASELINE config 3's model: clamped rods, n = 100, gravity along -y, no action
    n = 2048
    h = nat.Handle(model=nat.MODEL_ROD, n_env=n, n_elem=100, dt=5e-5, base_length=1.0, base_radius=0.025,
                   density=1000.0, youngs_modulus=1e6, gravity=(0, -9.80665, 0), damping_constant=2e-3,
                   bc_kind=nat.BC_ONE_END_FIXED, math=nat.MATH_FAST)
    ang = np.deg2rad(rng.uniform(-5, 5, n))
    init = np.zeros((n, 9))
    init[:, 3], init[:, 4], init[:, 6], init[:, 7] = np.cos(ang), np.sin(ang), -np.sin(ang), np.cos(ang)
    h.reset_host(init)
    steps, acts = 5, False
obs, rew, term, states = [], [], [], []
for s in range(steps):
    a = rng.uniform(-22, 22, (n, 1)).astype(np.float32) if acts else None
    o, r, t = h.step_host(a, 400)
    obs.append(o.copy()); rew.append(r.copy()); term.append(t.copy())
    if s in (0, steps - 1):
        states.append(h.state_tensor().cpu().numpy())
np.savez(out, obs=np.array(obs), rew=np.array(rew), term=np.array(term), state=np.array(states),
         fallback=h.fallback_count(), nonplanar=h.nonplanar_count())
h.close()
"""


def _run(tmp_path, case, planar):
    script = tmp_path / "planar_worker.py"
    script.write_text(_WORKER)
    out = tmp_path / f"{case}_{int(planar)}.npz"
    env = dict(os.environ)
    env.pop("SOFTROD_LEAN_PLANAR", None)
    if not planar:
        env["SOFTROD_LEAN_PLANAR"] = "0"
    res = subprocess.run([sys.executable, str(script), ROOT, case, str(out)], stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True, env=env, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:]
    return dict(np.load(out))


def _assert_same(a, b):
    for k in ("state", "obs", "rew", "term"):
        assert a[k].shape == b[k].shape, k
        assert np.array_equal(a[k], b[k]), (k, np.argwhere(a[k] != b[k])[:5])   # (-0.0 == 0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["pendulum", "clamped"])
def test_planar_kernel_gives_the_bits_of_the_3d_kernel(tmp_path, case):
    """4096 SoftPendulum envs (10 random-action steps) and 2048 clamped rods of n = 100 (5 steps): both are more items
    than resident CTA slots, so some items are split between two slots (stream-K hand-over).  Planar against 3D:
    equal state blocks after the first and the last step, equal outputs of every step, no fallback of any kind."""
    ref, pl = _run(tmp_path, case, False), _run(tmp_path, case, True)
    _assert_same(ref, pl)
    assert np.isfinite(pl["state"]).all()
    assert int(pl["fallback"]) == 0 and int(ref["fallback"]) == 0
    assert int(pl["nonplanar"]) == 0 and int(ref["nonplanar"]) == 0


@pytest.mark.gpu
def test_envs_out_of_the_plane_take_the_3d_kernel_without_a_range_fallback(tmp_path):
    """A SoftPendulum handle where one env is reset tilted out of the plane and two are pushed out of it through the
    state: every env matches the 3D path bit for bit, the planar kernel hands the three over as non-planar (counted
    apart from the range fallbacks, which stay at 0), and the handle then steps with the 3D pair."""
    ref, pl = _run(tmp_path, "mixed", False), _run(tmp_path, "mixed", True)
    _assert_same(ref, pl)
    assert int(pl["fallback"]) == 0 and int(ref["fallback"]) == 0
    assert int(ref["nonplanar"]) == 0
    # three envs, every step until the first poll of the counters moves the handle to the 3D pair (8 or 9 steps)
    assert 3 * 8 <= int(pl["nonplanar"]) <= 3 * 9, int(pl["nonplanar"])
    st = pl["state"][-1]
    assert all(np.abs(st[e, 2]).max() > 0 for e in (5, 9, 17))      # (they did leave the plane: x_z)


# ---- the planar rods of the GPU cases ----------------------------------------------------------------------------
def _rod_case(n):
    """The plain FP64 rod of shape n that use_planar accepts: the BC cycles through free / clamp / slider and the damper
    through on / off over the shape table (every combination twice), gravity lies in the x-y plane with |g_x| >= 2."""
    i = sorted(SHAPES).index(n)
    rng = np.random.default_rng(500 + n)
    while True:
        b = rng.uniform(0, 2 * np.pi)
        if abs(np.cos(b)) >= 0.2:
            break
    r, dt = (0.025, 1e-4) if n <= 50 else (0.025, 5e-5) if n <= 100 else (0.025, 2e-5) if n <= 200 else \
        (0.01, 1e-5) if n <= 300 else (0.008, 5e-6)
    return dict(n_elem=n, dt=dt, base_length=1.0, base_radius=r, density=1000.0, youngs_modulus=1e6,
                gravity=(9.80665 * np.cos(b), 9.80665 * np.sin(b), 0.0), damping_constant=2e-4 if (i // 3) % 2 == 0 else -1.0,
                bc_kind=(BC_FREE, BC_ONE_END_FIXED, BC_PENDULUM_SLIDER)[i % 3])


def _planar_init(rng, n_env):
    """sr_reset rows: start in the plane, direction at a random in-plane angle, normal turned +-90 degrees from it in the
    plane, so that d2 = direction x normal is +z or -z (config 3 has +z, SoftPendulum -z)."""
    a, s = rng.uniform(0, 2 * np.pi, n_env), rng.choice([-1.0, 1.0], n_env)
    init = np.zeros((n_env, 9))
    init[:, 0:2] = rng.uniform(-1, 1, (n_env, 2))
    init[:, 3], init[:, 4] = np.cos(a), np.sin(a)
    init[:, 6], init[:, 7] = -s * np.sin(a), s * np.cos(a)
    return init


def _tilt(init, env, phi):
    """Tilt env's rod phi out of the plane (the normal stays in the plane, orthogonal to the new direction)."""
    init[env, 3] *= np.cos(phi); init[env, 4] *= np.cos(phi); init[env, 5] = np.sin(phi)


def _planar_motion(rng, n_env, n):
    """Smooth in-plane node velocities and element rates w_1 (nodes / elements >= 1: the BCs pin the first), so that
    free rods deform too instead of falling rigidly."""
    s = np.linspace(0.0, 1.0, n + 1)
    c = rng.uniform(-1, 1, (n_env, 5))
    v = np.zeros((n_env, 3, n + 1))
    v[:, 0] = 0.1 * (c[:, 0:1] * np.sin(np.pi * s) + c[:, 1:2] * np.cos(2 * np.pi * s))
    v[:, 1] = 0.1 * c[:, 2:3] * np.sin(3 * np.pi * s)
    se = 0.5 * (s[1:] + s[:-1])
    w1 = 2.0 * (c[:, 3:4] * np.sin(np.pi * se) + c[:, 4:5] * np.cos(3 * np.pi * se))
    v[:, :, 0] = 0.0; w1[:, 0] = 0.0
    return v, w1


# ---- D: three envs that leave the fast-math range inside the plane ------------------------------------------------
RANGE = dict(n_elem=95, dt=5e-5, base_length=1.0, base_radius=0.025, density=1000.0, youngs_modulus=1e6,
             gravity=(1.5, -9.7, 0.0), damping_constant=2e-3, bc_kind=BC_ONE_END_FIXED)
RANGE_ENVS, RANGE_KINK, RANGE_SPIN, RANGE_STRETCH = 16, 3, 6, 9
RANGE_LAUNCHES = (5, 5, 5, 5)


def _lean_const(name):
    import re
    hdr = open(os.path.join(ROOT, "gym_softrobot_b200", "csrc", "rod_math.cuh")).read()
    return float(re.search(name + r"\s*=\s*([0-9.eE+-]+)", hdr).group(1))


def _stretch_limit(c):
    """The lean kernels' range of the damper map, e - 1 <= kLeanExpZ / |ln c_w|: the host's arithmetic (fill_args)."""
    PI, n, r = 3.141592653589793, c["n_elem"], c["base_radius"]
    rl = c["base_length"] / n
    A0 = PI * r * r
    J0 = A0 * A0 / (4.0 * PI) * (c["density"] * rl)
    mass = c["density"] * (PI * (r * r) * rl)
    return _lean_const("kLeanExpZ") / abs(-c["damping_constant"] * c["dt"] * mass * (1.0 / J0))


def _range_state(x, Q, w):
    """In place, on [env, ...] arrays of the clamped handle: env RANGE_KINK gets a 30 degree in-plane kink (frames of the
    outer half turned about d2 = +-z, nodes rebuilt along the turned d3), env RANGE_SPIN spins its last element about
    d2 at dt w_1 = 0.15 (> 0.1, the rotation map's range), env RANGE_STRETCH has its outer half stretched to twice the
    damper map's limit."""
    n, m = RANGE["n_elem"], RANGE["n_elem"] // 2
    t = np.deg2rad(30.0)
    Rz = np.array([[np.cos(t), -np.sin(t), 0.0], [np.sin(t), np.cos(t), 0.0], [0.0, 0.0, 1.0]])
    e = RANGE_KINK
    ln = np.sqrt(np.sum(np.diff(x[e], axis=1) ** 2, axis=0))
    for k in range(m, n):
        Q[e, :, :, k] = Q[e, :, :, k] @ Rz.T
        x[e, :, k + 1] = x[e, :, k] + ln[k] * Q[e, 2, :, k]
    w[RANGE_SPIN, 1, n - 1] = 0.15 / RANGE["dt"]
    e, f = RANGE_STRETCH, 1.0 + 2.0 * _stretch_limit(RANGE)
    dx = np.diff(x[e], axis=1)
    for k in range(m, n):
        x[e, :, k + 1] = x[e, :, k] + f * dx[:, k]


# ---- E: the non-planar window ------------------------------------------------------------------------------------
WINDOW_ENVS, WINDOW_PROBE, WINDOW_STEPS = 64, 7, 1100


def _window_counts(steps):
    """nonplanar_count() after each of `steps` one-substep steps with one tilted env (use_fast_pair, softrod_api.cu).
    The planar kernel flags the env at every step it runs.  At step 8k the handle fetches the counters (the copy is
    queued before step 8k's launch and sees steps 1..8k-1), and reads them at step 8k + 1: if more than 1 % of the
    window's 8 x 64 env-steps were handed over, steps 8k + 1 .. 8k + 512 take the 3D pair.  So steps 1-8 are planar
    (count 1..8, the fetch at step 8 sees 7 > 5.12), 9-520 are not (count stays 8), 521-528 are planar again (the fetch
    at step 520 saw nothing new; 9..16; the fetch at 528 sees 7 new), 529-1040 are not (16), 1041-1048 are (17..24),
    and so on: count(s) = 8 (s // 520) + min(s % 520, 8)."""
    s = np.arange(1, steps + 1)
    return 8 * (s // 520) + np.minimum(s % 520, 8)


# ---- the GPU worker --------------------------------------------------------------------------------------------------
_SHAPE_WORKER = r"""
import hashlib, os, sys
import numpy as np
root, cases, out = sys.argv[1], sys.argv[2].split(","), sys.argv[3]
sys.path[:0] = [root, os.path.join(root, "tests")]
import torch
import test_planar as tp
from gym_softrobot_b200 import _native as nat
from gym_softrobot_b200.envs.soft_pendulum import _make_handle, pendulum_init_params
sm = torch.cuda.get_device_properties(0).multi_processor_count
res = {}

def state(h):     # (+ 0.0: the 3D kernels may write -0.0 where the planar kernel keeps the reset's +0.0)
    return h.state_tensor().cpu().numpy() + 0.0

def counts(h):
    return np.array([h.fallback_count(), *h.fallback_causes(), h.nonplanar_count(), h.launch_count])

def init_fields(h):
    return np.concatenate([h.fields()[k].cpu().numpy().reshape(h.n_env, -1) for k in
                           ("position_collection", "velocity_collection", "director_collection", "omega_collection")], axis=1)

def run(key, h, launches, rng, full):
    # full: the state block after every launch; else one digest per env (batches of up to 1e5 envs)
    for li, k in enumerate(launches):
        a = rng.uniform(-22, 22, (h.n_env, 1)).astype(np.float32) if h.action_dim else None
        o, r, t = h.step_host(a, k)
        res[f"{key}/obs{li}"], res[f"{key}/rew{li}"], res[f"{key}/term{li}"] = o.copy(), r.copy(), t.copy()
        st = state(h)
        assert np.isfinite(st).all(), key
        res[f"{key}/state{li}"] = st if full else np.array([hashlib.blake2b(e.tobytes(), digest_size=16).digest() for e in st])
    res[f"{key}/counts"] = counts(h)

def batch_sizes(rods):   # too small to split / more items than resident slots (<= 2048 / 384 = 5 CTAs per SM)
    return (("small", 128), ("big", (5 * sm + 37) * rods))

if "shapes" in cases:
    for n, (nt, rods, _) in tp.SHAPES.items():
        c = tp._rod_case(n)
        for size, n_env in batch_sizes(rods):
            rng = np.random.default_rng(7 * n + n_env)
            h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, math=nat.MATH_FAST, **c)
            init = tp._planar_init(rng, n_env)
            tp._tilt(init, tp.PROBE, 0.01)
            h.reset_host(init)
            v, w1 = tp._planar_motion(rng, n_env, n)
            fl = h.fields()
            fl["velocity_collection"][:] = torch.as_tensor(v, device="cuda")
            fl["omega_collection"][:, 1] = torch.as_tensor(w1, device="cuda")
            torch.cuda.synchronize()     # (the handle steps on a stream of its own)
            if size == "small":
                res[f"rod{n}/small/init"] = init_fields(h)
            run(f"rod{n}/{size}", h, tp.LAUNCHES, rng, size == "small")
            h.close()
    for size, n_env in batch_sizes(15):      # SoftPendulum-v0's model at n = 32 (15 rods per CTA, warps shared by two)
        rng = np.random.default_rng(32 + n_env)
        h = _make_handle(n_env, 32, 1e-4, 0, nat.MATH_FAST)
        init = pendulum_init_params(rng.random(n_env))
        tp._tilt(init, tp.PROBE, 0.01)
        h.reset_host(init)
        run(f"pendulum/{size}", h, tp.LAUNCHES, rng, size == "small")
        h.close()
    h = nat.Handle(model=nat.MODEL_ROD, n_env=128, math=nat.MATH_FAST, **tp._rod_case(50))
    res["layout"] = np.array([getattr(h.state_view(), f) for f in ("f_position", "f_velocity", "f_director", "f_omega",
                                                                   "f_tangents", "f_kappa", "f_sigma", "f_dilatation")])
    h.close()

if "gz" in cases:     # rods in the x-y plane under gravity with a z component: not a planar problem
    c = dict(tp._rod_case(50), gravity=(1.0, -9.7, 2.5))
    h = nat.Handle(model=nat.MODEL_ROD, n_env=8, math=nat.MATH_FAST, **c)
    h.reset_host(tp._planar_init(np.random.default_rng(5), 8))
    res["gz/init"] = init_fields(h)
    run("gz", h, tp.LAUNCHES, None, True)
    h.close()

if "range" in cases:
    h = nat.Handle(model=nat.MODEL_ROD, n_env=tp.RANGE_ENVS, math=nat.MATH_FAST, **tp.RANGE)
    h.reset_host(tp._planar_init(np.random.default_rng(95), tp.RANGE_ENVS))
    fl = h.fields()
    x, Q, w = (fl[k].cpu().numpy() for k in ("position_collection", "director_collection", "omega_collection"))
    tp._range_state(x, Q, w)
    for k, a in (("position_collection", x), ("director_collection", Q), ("omega_collection", w)):
        fl[k][:] = torch.as_tensor(a, device="cuda")
    torch.cuda.synchronize()
    res["range/init"] = init_fields(h)
    run("range", h, tp.RANGE_LAUNCHES, None, True)
    h.close()

if "window" in cases:
    rng = np.random.default_rng(64)
    h = _make_handle(tp.WINDOW_ENVS, 50, 1e-4, 0, nat.MATH_FAST)
    init = pendulum_init_params(rng.random(tp.WINDOW_ENVS))
    tp._tilt(init, tp.WINDOW_PROBE, 0.01)
    h.reset_host(init)
    np_counts, digests, obs, rew, term = [], [], [], [], []
    for s in range(tp.WINDOW_STEPS):
        o, r, t = h.step_host(rng.uniform(-22, 22, (tp.WINDOW_ENVS, 1)).astype(np.float32), 1)
        obs.append(o.copy()); rew.append(r.copy()); term.append(t.copy())
        np_counts.append(h.nonplanar_count())
        digests.append(hashlib.blake2b(state(h).tobytes(), digest_size=16).digest())
    res.update({"window/nonplanar": np.array(np_counts), "window/digest": np.array(digests), "window/obs": np.array(obs),
                "window/rew": np.array(rew), "window/term": np.array(term), "window/counts": counts(h)})
    h.close()

np.savez(out, **res)
"""

# SOFTROD_* settings of a worker process -> the cases it runs
SETTINGS = {"planar": ({}, "shapes,gz,range,window"), "3d": ({"SOFTROD_LEAN_PLANAR": "0"}, "shapes,range,window"),
            "safe": ({"SOFTROD_FASTPATH": "0"}, "range")}


@pytest.fixture(scope="module")
def worker(tmp_path_factory):
    """setting -> the worker's results; each setting runs once per module, in a process of its own (the settings are
    read once per process)."""
    tmp = tmp_path_factory.mktemp("planar")
    script = tmp / "planar_worker.py"
    script.write_text(_SHAPE_WORKER)

    @functools.lru_cache(maxsize=None)
    def get(setting):
        extra, cases = SETTINGS[setting]
        env = {k: v for k, v in os.environ.items() if k not in ("SOFTROD_LEAN_PLANAR", "SOFTROD_FASTPATH")}
        env.update(extra)
        out = tmp / f"{setting}.npz"
        res = subprocess.run([sys.executable, str(script), ROOT, cases, str(out)], stdout=subprocess.PIPE,
                             stderr=subprocess.STDOUT, text=True, env=env, timeout=1800)
        assert res.returncode == 0, res.stdout[-3000:]
        return dict(np.load(out))
    return get


def _fields(st, layout, n):
    """The eight reference fields of one env's state block (Handle.fields)."""
    p, v, d, w, t, k, s, dl = layout
    return {"position_collection": st[p:p + 3, :n + 1], "velocity_collection": st[v:v + 3, :n + 1],
            "director_collection": st[d:d + 9, :n].reshape(3, 3, n), "omega_collection": st[w:w + 3, :n],
            "tangents": st[t:t + 3, :n], "kappa": st[k:k + 3, :n - 1], "sigma": st[s:s + 3, :n], "dilatation": st[dl, :n]}


def _oracle(c, init_row, fields0):
    """The C oracle's rod for a GPU env: built from the same sr_reset row, then given the env's x, v, Q, w as the
    GPU held them before the first launch (fields0: Handle.fields flattened, as the worker saves them)."""
    import rod_oracle as ro
    n = c["n_elem"]
    kw = {k: c[k] for k in ("gravity", "damping_constant", "bc_kind")}
    r = ro.OracleRod(n, init_row[0:3], init_row[3:6], init_row[6:9], c["base_length"], c["base_radius"], c["density"],
                     c["youngs_modulus"], c["dt"], **kw)
    sizes = (3 * (n + 1), 3 * (n + 1), 9 * n, 3 * n)
    parts = np.split(fields0, np.cumsum(sizes)[:-1])
    for name, a in zip(("position_collection", "velocity_collection", "director_collection", "omega_collection"), parts):
        getattr(r, name)[...] = a.reshape(getattr(r, name).shape)
    return r


def _assert_same_launches(a, b, key, launches):
    for li in range(launches):
        for f in ("state", "obs", "rew", "term"):
            x, y = a[f"{key}/{f}{li}"], b[f"{key}/{f}{li}"]
            assert x.shape == y.shape, (key, f)
            assert np.array_equal(x, y), (key, f, li, np.argwhere(x != y)[:5])      # (-0.0 == 0.0 in obs)


# ---- B -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", [f"rod{n}" for n in SHAPES] + ["pendulum"])
def test_planar_kernel_matches_3d_on_every_cta_shape(worker, case):
    """Every CTA shape of the planar kernel (SHAPES; SoftPendulum-v0's model at n = 32) against the 3D kernel, for a
    batch of 128 envs (too small to split) and one of more items than resident CTA slots (stream-K hand-over).  Per
    shape: BC, damper and in-plane gravity with g_x != 0 as _rod_case draws them, per env a random in-plane orientation,
    d2 = +z or -z and smooth in-plane motion.  Equal state blocks (stale slots n - 1 and n included) after each launch,
    equal outputs, no range fallback.  One env per batch (PROBE) is tilted 0.01 rad out of the plane: the planar
    kernel hands it to the 3D safe kernel once per launch, which shows that it ran the others."""
    ref, pl = worker("3d"), worker("planar")
    for size in ("small", "big"):
        key = f"{case}/{size}"
        _assert_same_launches(ref, pl, key, len(LAUNCHES))
        fb, causes, nonplanar, launches = ref[f"{key}/counts"][0], ref[f"{key}/counts"][1:4], ref[f"{key}/counts"][4], ref[f"{key}/counts"][5]
        assert fb == 0 and not causes.any() and nonplanar == 0, (key, ref[f"{key}/counts"])
        assert list(pl[f"{key}/counts"]) == [0, 0, 0, 0, len(LAUNCHES), launches], (key, pl[f"{key}/counts"])
        assert launches == 1 + 2 * len(LAUNCHES)          # reset + (fast-only, fallback) per launch


# ---- C -------------------------------------------------------------------------------------------------------------
ORACLE_FIELDS = ("position_collection", "velocity_collection", "director_collection", "omega_collection",
                 "tangents", "kappa", "sigma", "dilatation")


def _check_vs_oracle(res, key, c, init, envs, launches, what):
    """Envs `envs` of a worker case against the C oracle after every launch; returns the oracle's last fields."""
    from test_parity_gpu import assert_state_close, one_ulp_divergence, rate_floors
    n, layout = c["n_elem"], res["layout"]
    for e in envs:
        mk = lambda: _oracle(c, init[e], res[f"{key}/init"][e])
        o, refs = mk(), []
        for k in launches:
            o.substeps(k)
            refs.append({name: getattr(o, name).copy() for name in ORACLE_FIELDS})
        o.close()
        # the oracle's one-ulp divergence over the whole horizon (measured once per env, used at every launch)
        sens = one_ulp_divergence(mk, lambda rod: rod.substeps(sum(launches)), refs[-1])
        for li, ref in enumerate(refs):
            f = _fields(res[f"{key}/state{li}"][e], layout, n)
            x = ref["position_collection"]
            floors = rate_floors(c["youngs_modulus"], c["density"], c["base_length"], n, c["base_radius"], np.abs(x).max())
            for name in ORACLE_FIELDS:
                assert_state_close(f[name], ref[name], name, floors, f"{what} env {e} after launch {li}", measured=sens)
            obs = res[f"{key}/obs{li}"][e]
            np.testing.assert_allclose(obs[:3], x[:, -1], rtol=2e-6, atol=1e-7)
            np.testing.assert_allclose(obs[3:6], ref["velocity_collection"][:, -1], rtol=2e-6, atol=1e-7)
    return refs[-1]


@pytest.mark.gpu
@pytest.mark.parametrize("n", list(SHAPES))
def test_planar_rods_vs_c_oracle(worker, n):
    """The planar kernel's rods of the 128-env batch of every shape (three envs each) against the C oracle started
    from the same state: all eight fields, the strain observables that the planar kernel rebuilds for the last element
    and the tip included, and the tip in the observation, after 400 and 1000 substeps (two launches).  Tolerance: the
    1e-9 rule of test_parity_gpu with the oracle's own one-ulp divergence."""
    pl, c = worker("planar"), _rod_case(n)
    init = _planar_init(np.random.default_rng(7 * n + 128), 128)
    _check_vs_oracle(pl, f"rod{n}/small", c, init, (0, 2, 127), LAUNCHES, f"n={n} bc={c['bc_kind']}")


@pytest.mark.gpu
def test_rods_under_z_gravity_take_the_3d_kernel(worker):
    """use_planar refuses gravity with a z component: rods that start in the x-y plane under such gravity leave it, as
    the C oracle shows, and the planar kernel (which never applies g_z) must not see them (no env handed over as
    non-planar; it would have kept them flat)."""
    pl = worker("planar")
    c = dict(_rod_case(50), gravity=(1.0, -9.7, 2.5))
    init = _planar_init(np.random.default_rng(5), 8)
    last = _check_vs_oracle(pl, "gz", c, init, range(8), LAUNCHES, "g_z != 0")
    assert list(pl["gz/counts"][:5]) == [0, 0, 0, 0, 0], pl["gz/counts"]
    assert np.abs(last["position_collection"][2]).max() > 1e-3          # (they did leave the plane)


# ---- D -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_range_fallbacks_inside_the_plane(worker):
    """A clamped handle at n = 95 (4 rods per 384-thread CTA) with three envs that leave the fast-math range without
    leaving the plane (_range_state: a 30 degree bend, an in-plane spin at dt w_1 = 0.15, a stretch of twice the damper
    map's limit).  The planar kernel must flag them where the 3D kernel does — equal fallback counts and causes, each
    cause hit, none handed over as non-planar — and the state block must be equal to the 3D pair's and to the safe
    kernel's alone (SOFTROD_FASTPATH=0) after every launch.  Every env matches the C oracle.  4 launches of 5 substeps:
    the handle keeps the pair (the counters are first polled at step 8), and the spin stays within 20 substeps."""
    pl, ref, safe = worker("planar"), worker("3d"), worker("safe")
    L = len(RANGE_LAUNCHES)
    for other in (ref, safe):
        for li in range(L):
            assert np.array_equal(pl[f"range/state{li}"], other[f"range/state{li}"]), (li, np.argwhere(pl[f"range/state{li}"] != other[f"range/state{li}"])[:5])
            for f in ("obs", "rew", "term"):
                assert np.array_equal(pl[f"range/{f}{li}"], other[f"range/{f}{li}"]), (f, li)
    cp, cr = pl["range/counts"], ref["range/counts"]
    assert list(cp[:4]) == list(cr[:4]), (cp, cr)
    assert cp[1] > 0 and cp[2] > 0 and cp[3] > 0, cp                   # rotation, bend, stretch
    assert cp[4] == 0 and cr[4] == 0, (cp, cr)
    assert cp[5] == cr[5] == 1 + 2 * L and safe["range/counts"][5] == 1 + L
    init = _planar_init(np.random.default_rng(95), RANGE_ENVS)
    _check_vs_oracle(pl, "range", RANGE, init, range(RANGE_ENVS), RANGE_LAUNCHES, "range")


# ---- E -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_non_planar_window_ends(worker):
    """One SoftPendulum env of 64 is tilted out of the plane for good, and the handle steps 1100 times with one substep
    each: the planar kernel hands it over in bursts of 8 steps, separated by the 512 steps in which the handle uses
    the 3D pair (exact counts: _window_counts).  The state block (digest) and outputs equal the 3D process's at
    every step."""
    pl, ref = worker("planar"), worker("3d")
    assert np.array_equal(pl["window/nonplanar"], _window_counts(WINDOW_STEPS)), \
        np.flatnonzero(pl["window/nonplanar"] != _window_counts(WINDOW_STEPS))[:5]
    assert not ref["window/nonplanar"].any()
    for f in ("digest", "obs", "rew", "term"):
        bad = np.flatnonzero([not np.array_equal(a, b) for a, b in zip(pl[f"window/{f}"], ref[f"window/{f}"])])
        assert bad.size == 0, (f, "first step that differs", bad[:1] + 1)
    assert pl["window/counts"][0] == 0 and ref["window/counts"][0] == 0


# ---- A (CPU) -----------------------------------------------------------------------------------------------------------
def test_shape_table_follows_the_host_rule():
    """SHAPES against lean_threads_setting (softrod_api.cu) and the kernel's choice of barriers."""
    for n, (nt, rods, bar) in SHAPES.items():
        tpr = n + 1
        util = lambda t: (t // tpr) * tpr / t
        best = 512
        if util(384) > util(best) + 0.02:
            best = 384
        if util(256) > util(best) + 0.02:
            best = 256
        assert (best, best // tpr) == (nt, rods), n
        assert ("named" if tpr >= 32 and 2 <= rods <= 15 else "cta") == bar, n


@pytest.mark.parametrize("bc", [BC_FREE, BC_ONE_END_FIXED, BC_PENDULUM_SLIDER], ids=["free", "clamp", "slider"])
def test_oracle_keeps_planar_rods_in_their_plane(bc):
    """The premise of the planar kernel for every configuration use_planar accepts: clamped, free and slider rods at
    random in-plane orientations, with d2 = +z and -z, gravity with both in-plane components, with and without the
    damper, and moving in the plane, keep the eleven out-of-plane components exactly 0.0 over 3000 substeps.  The
    same rod under gravity with a z component leaves the plane."""
    import rod_oracle as ro
    rng = np.random.default_rng(30 + bc)
    for n, s, damp in ((7, 1.0, 2e-4), (31, -1.0, -1.0), (64, -1.0, 2e-3), (95, 1.0, -1.0)):
        a, b = rng.uniform(0, 2 * np.pi), rng.uniform(0.2, 1.3) * rng.choice([-1, 1]) + rng.choice([0.0, np.pi])
        start, d, nn = [*rng.uniform(-1, 1, 2), 0.0], [np.cos(a), np.sin(a), 0.0], [-s * np.sin(a), s * np.cos(a), 0.0]
        g = (9.80665 * np.cos(b), 9.80665 * np.sin(b), 0.0)      # (|b| >= 0.2 from both axes: g_x, g_y != 0)
        dt = 1e-4 if n <= 50 else 5e-5
        mk = lambda gz: ro.OracleRod(n, start, d, nn, 1.0, 0.025, 1000.0, 1e6, dt, gravity=(g[0], g[1], gz),
                                     damping_constant=damp, bc_kind=bc)
        r = mk(0.0)
        assert np.all(np.sign(r.director_collection[1, 2]) == s)          # d2 = +z / -z
        v, w1 = _planar_motion(rng, 1, n)
        r.velocity_collection[...] = v[0]
        r.omega_collection[1] = w1[0]
        for _ in range(6):
            r.substeps(500)
            _assert_in_plane(r, (n, s, damp))
        assert np.abs(r.velocity_collection[:2]).max() > 1e-2 and np.abs(r.omega_collection[1, 1:]).max() > 1e-2
        r.close()
        r = mk(2.5)
        r.substeps(3000)
        assert np.abs(r.position_collection[2]).max() > 1e-3
        r.close()
