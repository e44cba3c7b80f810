"""The planar model's trace check in the first substep of every segment (rod_kernel_lean.cuh, substep_planar's FIRST
copy).  A neighbour pair bent by 165 degrees in the plane has w^2 = 4 sin^2(165 deg) = 0.27, back inside the bend map's
range (kNarrowBendW2 = 0.6144, rod_math.cuh): only the trace check, which rules out a state that starts beyond 60 degrees
of bend, can flag it.

GPU: SoftPendulum-v0's model at n = 50 (15 rods per 768-thread CTA, per-rod named barriers) with a few envs kinked that
way, against the 3D pair (SOFTROD_LEAN_PLANAR=0), each in a subprocess of its own: equal state blocks, outputs and
fallback counts by cause after every launch.  The launches of 1, 3, 400 and 300 substeps run the segment that is the
item's last substep alone, segments of two and more substeps, and (in the batch of 4096 envs) segments that continue a
stream-K hand-over, some of which start at the item's last substep."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.abspath(os.path.dirname(__file__)))

RODS_PER_CTA = 15     # n = 50: 51 threads per rod in 768-thread CTAs
N_ENV = {"small": 128, "mid": 4096}   # 9 items, fewer than the slots: no split; 274 items: stream-K hand-overs
LAUNCHES = (1, 3, 400, 300)
KINK_DEG = 165.0


def kinked_envs(size, slots):
    """The kinked envs: rod 0 of an item (its warps hold one rod's barrier) and rod 1 (its first warp also holds rod
    0's end, so it takes two barriers).  In the split batch also the items whose second part, in the 3-substep launch,
    starts at substep 1 or at the last substep, as the fast-only launch's stream-K split of the items over `slots`
    (one 768-thread CTA per SM) gives them."""
    if size == "small":
        return [0, 16, 4 * RODS_PER_CTA + 1, 8 * RODS_PER_CTA]
    K = LAUNCHES[1]
    items = -(-N_ENV[size] // RODS_PER_CTA)
    cont = {}
    for p in range(1, slots):
        item, off = divmod(items * K * p // slots, K)
        cont.setdefault(off, item)
    return sorted({0, 16, 100 * RODS_PER_CTA, cont[1] * RODS_PER_CTA, cont[K - 1] * RODS_PER_CTA + 1,
                   (items - 2) * RODS_PER_CTA + 1})


_WORKER = r"""
import os, sys
import numpy as np
root, out = sys.argv[1], sys.argv[2]
sys.path[:0] = [root, os.path.join(root, "tests")]
import torch
import test_planar_first_substep as fs
from gym_softrobot_b200 import _native as nat
from gym_softrobot_b200.envs.soft_pendulum import _make_handle, pendulum_init_params
n, dt = 50, 1e-4
sm = torch.cuda.get_device_properties(0).multi_processor_count
res = {}
for size, n_env in fs.N_ENV.items():
    rng = np.random.default_rng(165 + n_env)
    h = _make_handle(n_env, n, dt, 0, nat.MATH_FAST)
    h.reset_host(pendulum_init_params(rng.random(n_env)))
    fl = h.fields()
    x, Q = (fl[k].cpu().numpy() for k in ("position_collection", "director_collection"))
    t = np.deg2rad(fs.KINK_DEG)   # outer half turned about d2 = +-z, nodes rebuilt along the turned d3
    Rz = np.array([[np.cos(t), -np.sin(t), 0.0], [np.sin(t), np.cos(t), 0.0], [0.0, 0.0, 1.0]])
    kinked = fs.kinked_envs(size, sm)
    res[size + "/kinked"] = np.array(kinked)
    for e in kinked:
        ln = np.sqrt(np.sum(np.diff(x[e], axis=1) ** 2, axis=0))
        for k in range(n // 2, n):
            Q[e, :, :, k] = Q[e, :, :, k] @ Rz.T
            x[e, :, k + 1] = x[e, :, k] + ln[k] * Q[e, 2, :, k]
    for k, a in (("position_collection", x), ("director_collection", Q)):
        fl[k][:] = torch.as_tensor(a, device="cuda")
    torch.cuda.synchronize()     # (the handle steps on a stream of its own)
    for li, k in enumerate(fs.LAUNCHES):
        a = rng.uniform(-22, 22, (n_env, 1)).astype(np.float32)
        o, r, te = h.step_host(a, k)
        key = f"{size}/{li}"
        res[key + "/obs"], res[key + "/rew"], res[key + "/term"] = o.copy(), r.copy(), te.copy()
        res[key + "/state"] = h.state_tensor().cpu().numpy() + 0.0   # (+ 0.0: -0.0 where the planar kernel keeps +0.0)
        res[key + "/counts"] = np.array([h.fallback_count(), *h.fallback_causes(), h.nonplanar_count(), h.launch_count])
    h.close()
np.savez(out, **res)
"""


def test_kinked_pair_is_inside_the_bend_map_but_fails_the_trace():
    """The premise: at 165 degrees w^2 is under kNarrowBendW2 with margin and the trace 1 + 2 cos(theta) is <= 2."""
    t = np.deg2rad(KINK_DEG)
    assert 4 * np.sin(t) ** 2 < 0.5 < 0.6144
    assert not (1 + 2 * np.cos(t) > 2.0)
    for size in N_ENV:
        for slots in (132, 148, 160):
            envs = kinked_envs(size, slots)
            assert max(envs) < N_ENV[size] and {e % RODS_PER_CTA for e in envs} == {0, 1}, (size, slots, envs)


@pytest.fixture(scope="module")
def worker(tmp_path_factory):
    """setting ("planar" or "3d") -> the worker's results, one process per setting (the switch is read once)."""
    tmp = tmp_path_factory.mktemp("planar_first")
    script = tmp / "worker.py"
    script.write_text(_WORKER)

    @functools.lru_cache(maxsize=None)
    def get(setting):
        env = {k: v for k, v in os.environ.items() if k not in ("SOFTROD_LEAN_PLANAR", "SOFTROD_FASTPATH")}
        if setting == "3d":
            env["SOFTROD_LEAN_PLANAR"] = "0"
        out = tmp / f"{setting}.npz"
        res = subprocess.run([sys.executable, str(script), ROOT, str(out)], stdout=subprocess.PIPE,
                             stderr=subprocess.STDOUT, text=True, env=env, timeout=1800)
        assert res.returncode == 0, res.stdout[-3000:]
        return dict(np.load(out))
    return get


@pytest.mark.gpu
@pytest.mark.parametrize("size", list(N_ENV))
def test_trace_check_flags_a_kink_beyond_the_bend_map_in_every_segment(worker, size):
    """The kinked envs are flagged for their bend in the one-substep launch (where nothing else can flag them) and
    re-run by the safe kernel; after every launch the state block, observations, rewards, terminations and the fallback
    counts by cause equal the 3D pair's."""
    pl, ref = worker("planar"), worker("3d")
    n_kinked = len(pl[f"{size}/kinked"])
    for li in range(len(LAUNCHES)):
        key = f"{size}/{li}"
        for f in ("state", "obs", "rew", "term"):
            a, b = pl[f"{key}/{f}"], ref[f"{key}/{f}"]
            assert a.shape == b.shape, (key, f)
            assert np.array_equal(a, b, equal_nan=True), (key, f, np.argwhere(a != b)[:5])
        cp, cr = pl[f"{key}/counts"], ref[f"{key}/counts"]
        assert list(cp[:4]) == list(cr[:4]), (key, cp, cr)
        assert cp[4] == cr[4] == 0, (key, cp, cr)                   # every env is planar
        assert cp[5] == cr[5], (key, cp, cr)
        if li == 0:
            assert cp[0] == cp[2] == n_kinked, (key, cp)            # the kinked envs, each for its bend
