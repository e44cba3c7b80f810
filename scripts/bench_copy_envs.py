"""Time env forks (sr_copy_envs) on the GPU: CUDA events around the call, 50 calls after warm-up, the median.

  a  4096 SoftPendulum-v0 envs (n = 50): env 0 onto the other 4095, within the handle (gather + scatter)
  b  the same handle: a random permutation of its 4096 envs (gather + scatter)
  c  a 1-env SoftPendulum handle onto every env of a 4096-env handle (one launch between handles)
  d  65 536 clamped rods (n = 100, bench.py config 3's rod): a random permutation
  e  16 384 8-arm x 40-element OctoFlat assemblies (bench.py config 4's): a random permutation

Bytes moved come from the per-env buffer table (csrc/softrod_api.cu: env_buffers): every copied row is read and
written once, twice over for a copy within one handle (through the staging buffer).  The rate over 7.7 TB/s (HBM3e of
one B200) is a share of HBM bandwidth only where the rows do not fit the 126 MB L2 (d, e).  For scale, one env-step
(the substeps of the handle's env-step: 400, and 401 for the OctoFlat env of e) of the destination handle,
with the count in each row.  Prints one JSON line per case, after the card's name, power limit and clock.
"""
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM_TBPS = 7.7
N_FIELDS, BC_DIM, AUX_DIM, HEAD_DIM = 32, 12, 8, 20   # csrc/rod_kernels.cuh


def main():
    import ctypes as C
    import torch
    from gym_softrobot_b200 import _native as nat
    from gym_softrobot_b200.envs.soft_pendulum import _make_handle, pendulum_init_params
    from gym_softrobot_b200.envs.octo_flat import OctoFlatVectorEnv

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps({"gpu": smi}), flush=True)
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(0)

    def rows(h, rest_kappa):
        """Bytes per env of the buffers sr_copy_envs moves for these handles: rod block, BC anchors, model scratch,
        head, and the rest curvature where allocated (env_buffers in csrc/softrod_api.cu)."""
        v = h.state_view()
        nr, st, es = h.n_rod, v.stride, v.elem_size
        return nr * N_FIELDS * st * es + nr * BC_DIM * es + AUX_DIM * es + HEAD_DIM * es + (nr * 3 * st * es if rest_kappa else 0)

    def time_copy(dst, src, d, s, calls=50, warmup=5):
        lib = dst._lib
        dt = torch.as_tensor(np.asarray(d, np.int32), device=dev)
        st = torch.as_tensor(np.asarray(s, np.int32), device=dev)
        stream = dst._stream_ptr()

        def call():
            nat._check(lib.sr_copy_envs(dst._h, C.c_void_p(dt.data_ptr()), src._h, C.c_void_p(st.data_ptr()), len(d), stream))
        for _ in range(warmup):
            call()
        torch.cuda.synchronize()
        ms = []
        for _ in range(calls):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); call(); e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        return float(np.median(ms)), float(np.min(ms)), float(np.max(ms))

    def time_step(h, action, K, reps=5):
        obs = torch.empty((h.n_env, max(h.obs_dim, 6)), dtype=torch.float32, device=dev)
        rew = torch.empty(h.n_env, dtype=torch.float64, device=dev)
        term = torch.empty(h.n_env, dtype=torch.uint8, device=dev)
        h.step(action, K, obs, rew, term)
        torch.cuda.synchronize()
        ms = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); h.step(action, K, obs, rew, term); e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        return float(np.median(ms))

    def report(case, what, n_pairs, per_env, staged, t, step_ms, step_substeps, fits_l2):
        moved = n_pairs * per_env * (4 if staged else 2)
        gbs = moved / (t[0] * 1e-3) / 1e9
        print(json.dumps({"case": case, "copy": what, "pairs": n_pairs, "bytes_per_env": per_env,
                          "bytes_moved": moved, "median_ms": round(t[0], 4), "min_ms": round(t[1], 4),
                          "max_ms": round(t[2], 4), "GB_per_s": round(gbs, 1),
                          "share_of_7.7TB_per_s": round(gbs / (HBM_TBPS * 1e3), 3),
                          "rows_fit_L2": fits_l2, "env_step_ms": round(step_ms, 3), "env_step_substeps": step_substeps}), flush=True)

    # a, b, c: SoftPendulum-v0, 4096 envs
    N = 4096
    pend = _make_handle(N, 50, 1e-4, 0, nat.MATH_FAST)
    pend.reset_host(pendulum_init_params(rng.random(N)))
    act = torch.as_tensor(rng.uniform(-22, 22, (N, 1)).astype(np.float32), device=dev)
    K = 400
    step_ms = time_step(pend, act, K)
    per_env = rows(pend, False)
    t = time_copy(pend, pend, np.arange(1, N), np.zeros(N - 1, int))
    report("a", "env 0 onto the other 4095 envs of the handle", N - 1, per_env, True, t, step_ms, K, True)
    perm = rng.permutation(N)
    t = time_copy(pend, pend, np.arange(N), perm)
    report("b", "a random permutation of the handle's 4096 envs", N, per_env, True, t, step_ms, K, True)
    one = _make_handle(1, 50, 1e-4, 0, nat.MATH_FAST)
    one.reset_host(pendulum_init_params(rng.random(1)))
    t = time_copy(pend, one, np.arange(N), np.zeros(N, int))
    report("c", "a 1-env handle onto every env of a 4096-env handle", N, per_env, False, t, step_ms, K, True)
    pend.close(); one.close()

    # d: 65 536 clamped rods, n = 100
    N = 65536
    rod = nat.Handle(model=nat.MODEL_ROD, n_env=N, n_elem=100, dt=5e-5, base_length=1.0, base_radius=0.025, density=1000.0,
                     youngs_modulus=1e6, gravity=(0, -9.80665, 0), damping_constant=2e-3, bc_kind=nat.BC_ONE_END_FIXED)
    ang = np.deg2rad(rng.uniform(-5, 5, N))
    init = np.zeros((N, 9))
    init[:, 3], init[:, 4], init[:, 6], init[:, 7] = np.cos(ang), np.sin(ang), -np.sin(ang), np.cos(ang)
    rod.reset_host(init)
    K = 400
    step_ms = time_step(rod, None, K)
    per_env = rows(rod, False)
    t = time_copy(rod, rod, np.arange(N), rng.permutation(N))
    report("d", "a random permutation of 65 536 clamped rods (n = 100)", N, per_env, True, t, step_ms, K, False)
    rod.close()

    # e: 16 384 OctoFlat assemblies of 8 arms x 40 elements (rest curvature allocated by reset)
    N = 16384
    env = OctoFlatVectorEnv(N, n_elems=40, time_step=3e-5, recording_fps=83, autoreset=False)
    env.reset(seed=42)
    K = env.step_skip
    step_ms = time_step(env.handle, None, K)
    per_env = rows(env.handle, True)
    t = time_copy(env.handle, env.handle, np.arange(N), rng.permutation(N))
    report("e", "a random permutation of 16 384 8 x 40 assemblies", N, per_env, True, t, step_ms, K, False)
    env.close()


if __name__ == "__main__":
    main()
