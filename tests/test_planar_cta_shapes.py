"""CTA shapes of the planar model's fast-only kernel (planar_threads_setting, softrod_api.cu): 768 threads where they
hold 2-15 rods of >= 32 threads, the lean kernel's CTA (lean_threads_setting) otherwise.  The 3D pair and the safe fallback keep the lean kernel's CTA in any case.

CPU: the rule as a table.
GPU: SoftPendulum-v0's model at n = 50 (15 rods per 768-thread CTA) against the 3D pair (SOFTROD_LEAN_PLANAR=0), each
in a subprocess of its own: equal state blocks, outputs and fallback counts after every launch; and the launches of
BASELINE config 2's handle under torch.profiler."""
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.abspath(os.path.dirname(__file__)))

# n_elem -> (threads of the planar kernel's CTA, rods per CTA, barriers).  31 / 32: 24 / 23 rods would fit 768 threads,
# past the 15 named barriers; 46 / 47: 16 rods of 47 / 48 threads, 384 threads as lean_threads_setting picks; 48 / 50:
# 15 rods; 100: 7 x 101 = 707 / 768 lanes (against 5 x 101 = 505 / 512); 383: two rods; 384: one rod.
PLANAR_SHAPES = {3: (512, 128, "cta"), 31: (512, 16, "cta"), 32: (512, 15, "named"), 46: (384, 8, "named"),
                 47: (384, 8, "named"), 48: (768, 15, "named"), 50: (768, 15, "named"), 95: (768, 8, "named"),
                 100: (768, 7, "named"), 160: (768, 4, "named"), 255: (768, 3, "named"), 256: (768, 2, "named"),
                 383: (768, 2, "named"), 384: (512, 1, "cta")}


def _lean_threads(n):
    """lean_threads_setting (softrod_api.cu) for rods of <= 511 elements."""
    tpr = n + 1
    util = lambda t: (t // tpr) * tpr / t
    best = 512
    if util(384) > util(best) + 0.02:
        best = 384
    if util(256) > util(best) + 0.02:
        best = 256
    return best


def _named(tpr, rods):   # per-rod named barriers (rod_kernel_lean.cuh)
    return tpr >= 32 and 2 <= rods <= 15


def _planar_threads(n):
    tpr = n + 1
    return 768 if _named(tpr, 768 // tpr) else _lean_threads(n)


def test_planar_shape_table_follows_the_host_rule():
    for n, (nt, rods, bar) in PLANAR_SHAPES.items():
        got = _planar_threads(n)
        assert (got, got // (n + 1)) == (nt, rods), n
        assert ("named" if _named(n + 1, rods) else "cta") == bar, n


# ---- GPU ---------------------------------------------------------------------------------------------------------------
PROBE, KINK, SPIN = 1, 5, 9     # envs of every batch: tilted out of the plane; kinked by 30 degrees; last element spun
LAUNCHES = (5, 400, 300)

_WORKER = r"""
import os, sys
import numpy as np
root, out = sys.argv[1], sys.argv[2]
sys.path[:0] = [root, os.path.join(root, "tests")]
import torch
import test_planar as tp
import test_planar_cta_shapes as cs
from gym_softrobot_b200 import _native as nat
from gym_softrobot_b200.envs.soft_pendulum import _make_handle, pendulum_init_params
sm = torch.cuda.get_device_properties(0).multi_processor_count
n, dt = 50, 1e-4
res = {}
# 128 envs: 9 items, no split; 4096: 273 items of 15 and one of a single env, more than the resident slots (stream-K
# hand-overs); and about five items per slot
for size, n_env in (("small", 128), ("mid", 4096), ("big", (5 * sm + 37) * 15)):
    rng = np.random.default_rng(50 + n_env)
    h = _make_handle(n_env, n, dt, 0, nat.MATH_FAST)
    init = pendulum_init_params(rng.random(n_env))
    tp._tilt(init, cs.PROBE, 0.01)
    h.reset_host(init)
    fl = h.fields()
    x, Q, w = (fl[k].cpu().numpy() for k in ("position_collection", "director_collection", "omega_collection"))
    t = np.deg2rad(30.0)      # outer half of env KINK turned about d2 = +-z, nodes rebuilt along the turned d3
    Rz = np.array([[np.cos(t), -np.sin(t), 0.0], [np.sin(t), np.cos(t), 0.0], [0.0, 0.0, 1.0]])
    ln = np.sqrt(np.sum(np.diff(x[cs.KINK], axis=1) ** 2, axis=0))
    for k in range(n // 2, n):
        Q[cs.KINK, :, :, k] = Q[cs.KINK, :, :, k] @ Rz.T
        x[cs.KINK, :, k + 1] = x[cs.KINK, :, k] + ln[k] * Q[cs.KINK, 2, :, k]
    w[cs.SPIN, 1, n - 1] = 0.12 / dt          # dt w_1 = 0.12 rad per substep, past the rotation map's 0.1
    for k, a in (("position_collection", x), ("director_collection", Q), ("omega_collection", w)):
        fl[k][:] = torch.as_tensor(a, device="cuda")
    torch.cuda.synchronize()     # (the handle steps on a stream of its own)
    for li, k in enumerate(cs.LAUNCHES):
        a = rng.uniform(-22, 22, (n_env, 1)).astype(np.float32)
        o, r, te = h.step_host(a, k)
        key = f"{size}/{li}"
        res[key + "/obs"], res[key + "/rew"], res[key + "/term"] = o.copy(), r.copy(), te.copy()
        res[key + "/state"] = h.state_tensor().cpu().numpy() + 0.0   # (+ 0.0: -0.0 where the planar kernel keeps +0.0)
        res[key + "/counts"] = np.array([h.fallback_count(), *h.fallback_causes(), h.nonplanar_count(), h.launch_count])
    h.close()
np.savez(out, **res)
"""


@pytest.fixture(scope="module")
def worker(tmp_path_factory):
    """setting ("planar" or "3d") -> the worker's results, one process per setting (the switch is read once)."""
    tmp = tmp_path_factory.mktemp("planar_cta")
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
@pytest.mark.parametrize("size", ["small", "mid", "big"])
def test_768_thread_planar_kernel_gives_the_bits_of_the_3d_pair(worker, size):
    """SoftPendulum-v0's model at n = 50 with one env tilted out of the plane (the planar kernel hands it to the safe
    kernel at every launch) and two that leave the fast-math range (a 30 degree kink, a spin past the rotation map):
    the state block, observations, rewards and terminations after every launch equal the 3D pair's, and so do the
    fallback counts by cause."""
    pl, ref = worker("planar"), worker("3d")
    for li in range(len(LAUNCHES)):
        key = f"{size}/{li}"
        for f in ("state", "obs", "rew", "term"):
            a, b = pl[f"{key}/{f}"], ref[f"{key}/{f}"]
            assert a.shape == b.shape, (key, f)
            assert np.array_equal(a, b, equal_nan=True), (key, f, np.argwhere(a != b)[:5])
        cp, cr = pl[f"{key}/counts"], ref[f"{key}/counts"]
        assert list(cp[:4]) == list(cr[:4]), (key, cp, cr)
        assert cp[0] > 0, (key, cp)                                # the range envs were re-run
        assert cp[4] == li + 1 and cr[4] == 0, (key, cp, cr)        # the tilted env, once per launch
        assert cp[5] == cr[5] == 1 + 2 * (li + 1), (key, cp, cr)    # reset + (fast-only, fallback) per launch


@pytest.mark.gpu
def test_config2_launches(tmp_path):
    """BASELINE config 2's handle (SoftPendulum-v0, 4096 envs, n = 50) under torch.profiler: the planar fast-only kernel
    launches 768-thread CTAs, one per resident slot (one per SM: 274 items of 15 envs are more than the slots), and the
    fallback launch 512-thread CTAs of the 3D safe kernel, one per item of 10 envs."""
    import torch
    sys.path.insert(0, ROOT)
    import gym_softrobot_b200 as g
    from torch.profiler import ProfilerActivity, profile

    n_env = 4096
    env = g.make_vec("SoftPendulum-v0", n_env, autoreset=False)
    env.reset(seed=42)
    a = (torch.rand((n_env, 1), device="cuda") * 44 - 22).float()
    env.handle.step(a, 400, env.obs, env.reward, env.terminated)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            env.handle.step(a, 400, env.obs, env.reward, env.terminated)
        torch.cuda.synchronize()
    env.close()
    trace = tmp_path / "trace.json"
    prof.export_chrome_trace(str(trace))
    kernels = [e for e in json.loads(trace.read_text())["traceEvents"]
               if e.get("cat") == "kernel" and "rod_lean_kernel" in e.get("name", "")]
    shapes = {(e["name"], tuple(e["args"]["grid"]), tuple(e["args"]["block"])) for e in kernels}
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    fast = [s for s in shapes if "rod_lean_kernel<double, 768, 1, true, (sr::LeanModel)6" in s[0]]
    safe = [s for s in shapes if "rod_lean_kernel<double, 512, 1, false, (sr::LeanModel)0" in s[0]]
    assert len(kernels) == 6 and len(shapes) == 2, shapes
    assert [s[1:] for s in fast] == [((sm, 1, 1), (768, 1, 1))], shapes
    assert [s[1:] for s in safe] == [(((n_env + 9) // 10, 1, 1), (512, 1, 1))], shapes
