"""Long rods on thread-block clusters (the cluster layout of rod_kernel_lean.cuh): device time per launch of K = 100
substeps.

Clamped rods (BASELINE config 3's model, the plain model), or with --model pendulum3d SoftPendulum3D-v0's rod (the
filter model: Laplace filter and moving base, base held still, 608 FLOP per element-substep), with --model contact a
free rod resting on a +z frictional plane with rest curvature, forcing first (OctoArmSingle's plane and friction, the
plane model: 720 FLOP per element-substep), with --model snake the same on a +y plane with the travelling-wave muscle
(the muscle model: 840), with --model spline SoftArmTracking-v0's clamped arm with its spline torques scaled by
40 / n (the spline model: 460), new random targets before every launch so that each launch pays one re-fit; at 2047
and 4095 elements it also times, alternating, unchanged targets (no re-fit) and new targets under a rate limit of
0.001 per substep, which keeps the re-fit running in every substep of the launch.  Each case has enough envs that the
state block exceeds the 126 MB L2 (>= 256 MB).
Cases: n = 600 and 1023 (SoftPendulum3D: 600 and 767, whose one-CTA kernel ends at 768 threads; 1023 on the cluster
kernel alone) on the one-CTA kernel (768 / 1024 threads) and on the forced cluster kernel (C = 2), which
run as alternating subprocesses (SOFTROD_LEAN_CLUSTER is read once per process), two rounds each; n = 1024, 2047 and
4095, where the cluster kernel is the only one.  Reported: ms per launch (median of 20 CUDA-event-timed launches after
warm-up), element-substeps/s, and the share of the measured FP64 peak (sr_measure_fp64_peak) at 440 FLOP per
element-substep (608 for SoftPendulum3D, and the models' counts above).  A probe compiled into a temporary directory reports how many clusters of C one-CTA-per-SM blocks
(512 threads, > 114 KB of shared memory each) the device keeps resident, and so what fraction of the SMs a full wave
of C-CTA clusters leaves idle.

    python scripts/bench_long_rods.py [--model rod|pendulum3d|contact|snake|spline] [--out FILE]   (the report goes to stdout, and to FILE if given)
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K, TIMED, WARMUP = 100, 20, 5
FLOP_PER_ELEMENT_SUBSTEP = {"rod": 440, "pendulum3d": 608, "contact": 720, "snake": 840, "spline": 460}
STATE_BYTES = 256 << 20
SPLINE_ROWS = {0: ", unchanged targets", 1: ", new targets every launch", 2: ", new targets every launch, rate-limited"}

_PROBE = r"""
#include <cstdio>
#include <cuda_runtime.h>
__global__ void __launch_bounds__(512, 1) probe(int *p) { extern __shared__ int s[]; if (p) p[threadIdx.x] = s[threadIdx.x]; }
int main() {
  const int smem = 120 * 1024;   // one CTA per SM, like the lean kernel's 512 threads x 128 registers
  if (cudaFuncSetAttribute(probe, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) return 1;
  for (int c = 1; c <= 8; c++) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(c); cfg.blockDim = dim3(512); cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute a; a.id = cudaLaunchAttributeClusterDimension;
    a.val.clusterDim.x = c; a.val.clusterDim.y = 1; a.val.clusterDim.z = 1;
    cfg.attrs = &a; cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, probe, &cfg) != cudaSuccess) return 2;
    printf("%d %d\n", c, n);
  }
  return 0;
}
"""


def one(n, cluster, model, refit):
    """Runs in a subprocess of its own: time one case, print one JSON line.  refit (spline model): 0 unchanged targets,
    1 new random targets before every launch, 2 the same under a rate limit that re-fits in every substep."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    from gym_softrobot_b200 import _native as nat
    stride = 32 * ((n + 1 + 31) // 32)
    n_env = -(-STATE_BYTES // (32 * stride * 8))
    act, new_targets = None, lambda: None
    assert model in FLOP_PER_ELEMENT_SUBSTEP, model
    if model == "pendulum3d":
        from gym_softrobot_b200.envs.soft_pendulum_3d import _make_handle, pendulum3d_init_params
        h = _make_handle(n_env, n, 2e-6 * 1023 / n, K, 0)
        h.reset_host(pendulum3d_init_params(np.random.default_rng(n).uniform(-1, 1, n_env)))
        act = torch.zeros((n_env, 2), dtype=torch.float32, device="cuda")
    elif model in ("contact", "snake"):
        from gym_softrobot_b200.envs.arm_single import arm_contact_params
        r0, normal = 0.004, np.array([0.0, 0.0, 1.0] if model == "contact" else [0.0, 1.0, 0.0])
        c = arm_contact_params()
        c["plane_origin"], c["plane_normal"] = list(-r0 * normal), list(normal)
        mus = dict(period=1.0, ramp_up_time=5e-4, phase_shift=0.7, direction=list(normal)) if model == "snake" else None
        h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n, dt=2e-6 * 1023 / n, base_length=1.0, base_radius=r0,
                       density=1000.0, youngs_modulus=1e6, gravity=tuple(-9.81 * normal), damping_constant=1e-2,
                       bc_kind=nat.BC_FREE, math=nat.MATH_FAST, contact=c, muscle=mus)
        axis = np.array([0.0, 1.0, 0.0] if model == "contact" else [0.0, 0.0, -1.0])
        h.reset_host(np.tile(np.concatenate([np.zeros(3), axis, normal]), (n_env, 1)))
        rk = np.random.default_rng(n).uniform(-3, 3, (n_env, 1)) * np.sin(3 * np.pi * np.linspace(0.0, 1.0, n - 1))[None, :]
        h.rest_kappa_tensor()[:, 0, :] = torch.as_tensor(rk, device="cuda")
        if mus:
            mu = h.muscle_tensor()
            mu[:, 1] = 6.0
            mu[:, 2:] = torch.as_tensor(2e-4 * np.sin(np.pi * np.linspace(0.0, 1.0, n)), device="cuda")
        torch.cuda.synchronize()
    elif model == "spline":
        from gym_softrobot_b200.envs.soft_arm_tracking import _E, _L, _N_CTRL, _R, spline_scale
        # the env's arm (_make_handle), with the rate limit of the case; 5e-6 s at 2048 elements
        h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n, dt=1e-5 * 1024 / n, base_length=_L, base_radius=_R,
                       density=1000 * 1e-6, youngs_modulus=_E, damping_constant=_E * 1e-7, bc_kind=nat.BC_ONE_END_FIXED,
                       damping_before_constraints=True,
                       spline=dict(directions=(0, 1), n_ctrl=_N_CTRL, scale=spline_scale(n),
                                   max_rate=1e-3 if refit == 2 else float("inf")))
        init = np.zeros((n_env, 9)); init[:, 4] = 1.0; init[:, 8] = 1.0      # the env's arm: along +y, normal +z
        h.reset_host(init)
        pts, _ = h.spline_tensors()
        gen = torch.Generator(device="cuda").manual_seed(n)

        def new_targets():
            pts[:, :2, :4] = torch.rand((n_env, 2, 4), generator=gen, dtype=torch.float64, device="cuda") * 2 - 1
        new_targets()
        torch.cuda.synchronize()
    else:   # rod
        h = nat.Handle(model=nat.MODEL_ROD, n_env=n_env, n_elem=n, dt=2e-6 * 1023 / n, base_length=1.0,
                       base_radius=0.004, density=1000.0, youngs_modulus=1e6, gravity=(0.0, -9.80665, 0.0),
                       damping_constant=2e-3, bc_kind=nat.BC_ONE_END_FIXED, math=nat.MATH_FAST)
        ang = np.deg2rad(np.random.default_rng(n).uniform(-5, 5, n_env))
        init = np.zeros((n_env, 9))
        init[:, 3], init[:, 4], init[:, 6], init[:, 7] = np.cos(ang), np.sin(ang), -np.sin(ang), np.cos(ang)
        h.reset_host(init)
    obs = torch.empty((n_env, h.obs_dim), dtype=torch.float32, device="cuda")
    rew = torch.empty(n_env, dtype=torch.float64, device="cuda")
    term = torch.empty(n_env, dtype=torch.uint8, device="cuda")
    s = torch.cuda.current_stream()
    for _ in range(WARMUP):
        if refit:
            new_targets()
        h.step(act, K, obs, rew, term)
    torch.cuda.synchronize()
    times = []
    for _ in range(TIMED):
        if refit:
            new_targets()   # (outside the timed window)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        h.step(act, K, obs, rew, term)
        e1.record(s)
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    assert np.isfinite(h.state_tensor().cpu().numpy()).all() and int(term.sum()) == 0
    ms = float(np.median(times))
    rate = n_env * n * K / (ms * 1e-3)
    print(json.dumps(dict(n=n, kernel="cluster" if cluster else "one-CTA", C=(n + 512) // 512 if cluster else 1, refit=refit,
                          n_env=n_env, state_MB=round(n_env * 32 * stride * 8 / 2**20), ms=ms, ms_min=min(times),
                          ms_max=max(times), elem_substeps_per_s=rate, fallbacks=h.fallback_count())))
    h.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the report to this file")
    ap.add_argument("--model", choices=sorted(FLOP_PER_ELEMENT_SUBSTEP), default="rod")
    ap.add_argument("--one", nargs=3, type=int, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.one:
        n, cluster, refit = a.one
        return one(n, cluster, a.model, refit)
    import torch
    sys.path.insert(0, ROOT)
    from gym_softrobot_b200 import _native as nat
    assert torch.cuda.is_available(), "this benchmark needs the GPU"
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    say(f"model: {a.model}; device: {torch.cuda.get_device_name(0)}, {sm} SMs; nvidia-smi name, power limit, max SM "
        f"clock, SM clock: {smi}")
    peak = nat.measure_fp64_peak(0)
    say(f"measured FP64 peak (sr_measure_fp64_peak): {peak:.2f} TFLOP/s")
    with tempfile.TemporaryDirectory() as tmp:
        src, exe = os.path.join(tmp, "probe.cu"), os.path.join(tmp, "probe")
        open(src, "w").write(_PROBE)
        nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", src, "-o", exe], check=True)
        for line in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split("\n"):
            if line.strip():
                c, nc = map(int, line.split())
                say(f"clusters of {c} one-CTA-per-SM blocks resident at once: {nc} ({nc * c} of {sm} SMs busy, "
                    f"{100.0 * (sm - nc * c) / sm:.1f} % idle)")
    if a.model in ("rod", "contact", "snake", "spline"):
        cases = [(600, 0), (600, 1), (1023, 0), (1023, 1)] * 2 + [(1024, 1), (2047, 1), (4095, 1)]
    else:    # (the filter model's largest CTA is 768 threads: from 768 elements on the cluster layout is the only one)
        cases = [(600, 0), (600, 1), (767, 0), (767, 1)] * 2 + [(1023, 1), (1024, 1), (2047, 1), (4095, 1)]
    cases = [(n, cl, 1) for n, cl in cases]
    if a.model == "spline":   # what the re-fit costs: none, one per launch, one in every substep (rate limited)
        cases += [(n, 1, refit) for n in (2047, 4095) for refit in (0, 1, 2)] * 2 + [(1023, 0, 2), (1023, 1, 2)] * 2
    for n, cl, refit in cases:
        env = dict(os.environ)
        env.pop("SOFTROD_LEAN_CLUSTER", None)
        if cl:
            env["SOFTROD_LEAN_CLUSTER"] = "1"
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--model", a.model, "--one", str(n), str(cl), str(refit)], env=env,
                             capture_output=True, text=True)
        if out.returncode != 0:
            raise SystemExit(out.stdout + out.stderr)
        r = json.loads(out.stdout.strip().splitlines()[-1])
        share = r["elem_substeps_per_s"] * FLOP_PER_ELEMENT_SUBSTEP[a.model] / (peak * 1e12)
        say(f"n={r['n']:5d} {r['kernel']:8s} C={r['C']} n_env={r['n_env']:5d} state={r['state_MB']} MB"
            f"{'' if a.model != 'spline' else SPLINE_ROWS[refit]}: "
            f"{r['ms']:.3f} ms/launch (min {r['ms_min']:.3f}, max {r['ms_max']:.3f}), "
            f"{r['elem_substeps_per_s'] / 1e9:.2f} G element-substeps/s, {100 * share:.1f} % of FP64 peak, "
            f"fallbacks {r['fallbacks']}")
    if a.out:
        open(a.out, "w").write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
