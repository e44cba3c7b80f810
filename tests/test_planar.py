"""The planar variant of the lean kernel (CVAR 8, rod_kernel_lean.cuh): rods that stay in the lab x-y plane are stepped
with the out-of-plane terms left out, and must give the bits of the 3D kernels (DESIGN.md §5).

CPU: the C oracle keeps every out-of-plane component of SoftPendulum-v0 an exact zero (the premise of the variant).
GPU: each case runs twice in a subprocess, with SOFTROD_LEAN_PLANAR=0 (3D kernels) and by default (planar), and the
whole state block, observations, rewards and termination flags must be equal."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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
            Q = r.director_collection
            for name, a in {"x_z": r.position_collection[2], "v_z": r.velocity_collection[2], "d1_z": Q[0, 2],
                            "d3_z": Q[2, 2], "d2_xy": Q[1, :2], "w_0": r.omega_collection[0],
                            "w_2": r.omega_collection[2], "kappa_02": r.kappa[[0, 2]], "sigma_1": r.sigma[1]}.items():
                assert np.all(a == 0.0), (seed, name, float(np.abs(a).max()))
        assert np.abs(r.omega_collection[1]).max() > 1e-3 and np.abs(r.velocity_collection[:2]).max() > 1e-3


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
