"""ctypes binding of the C-ABI in include/softrod.h (libsoftrod.so).

This is the only door to the physics: there is no CPU fallback.  If the CUDA
library is missing the import fails loudly; if there is no GPU, `sr_create`
returns SR_E_NO_DEVICE and `Handle` raises.
"""
import ctypes as C
import os

import numpy as np

from . import build as _build

SR_OK = 0
MODEL_ROD, MODEL_SOFT_PENDULUM, MODEL_SOFT_PENDULUM_3D = 0, 1, 2
BC_FREE, BC_ONE_END_FIXED, BC_PENDULUM_SLIDER, BC_MOVING_BASE = 0, 1, 2, 3
DTYPE_F64, DTYPE_F32 = 0, 1
MATH_FAST, MATH_FAITHFUL = 0, 1

# every symbol include/softrod.h declares (checked by tests/test_cabi.py)
EXPORTED_SYMBOLS = [
    "sr_abi_version", "sr_last_error", "sr_create", "sr_destroy", "sr_obs_dim", "sr_action_dim",
    "sr_init_dim", "sr_reset", "sr_step", "sr_reset_host", "sr_step_host", "sr_observe",
    "sr_get_state", "sr_set_state", "sr_copy_from", "sr_copy_envs", "sr_get_aux", "sr_get_head", "sr_get_rest_kappa", "sr_get_sucker", "sr_get_sucker_index", "sr_get_tm_activation", "sr_get_muscle_activation", "sr_get_fixed_suckers", "sr_get_ext_loads", "sr_get_muscle", "sr_get_spline", "sr_spline_basis", "sr_launch_count", "sr_fallback_count", "sr_fallback_causes", "sr_nonplanar_count", "sr_measure_fp64_peak", "sr_measure_fp64_peak_regs", "sr_selftest_reciprocals", "sr_probe_latency",
]


class SrConfig(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("device", C.c_int32), ("model", C.c_int32), ("dtype", C.c_int32),
        ("math", C.c_int32), ("n_env", C.c_int32), ("n_elem", C.c_int32), ("bc_kind", C.c_int32),
        ("point_force_on_base", C.c_int32), ("damping_before_constraints", C.c_int32),
        ("laplace_filter_order", C.c_int32), ("n_rod_per_env", C.c_int32),
        ("dt", C.c_double), ("base_length", C.c_double), ("base_radius", C.c_double),
        ("density", C.c_double), ("youngs_modulus", C.c_double), ("shear_modulus", C.c_double),
        ("gravity", C.c_double * 3), ("damping_constant", C.c_double),
        ("base_step", C.c_double), ("base_limit", C.c_double), ("base_move_period", C.c_double),
        ("contact_on", C.c_int32), ("contact_before_forcing", C.c_int32),
        ("plane_origin", C.c_double * 3), ("plane_normal", C.c_double * 3),
        ("contact_k", C.c_double), ("contact_nu", C.c_double), ("slip_velocity_tol", C.c_double),
        ("surface_tol", C.c_double), ("static_mu", C.c_double * 3), ("kinetic_mu", C.c_double * 3),
        ("has_head", C.c_int32), ("reserved1", C.c_int32),
        ("head_length", C.c_double), ("head_radius", C.c_double), ("head_density", C.c_double),
        ("joint_k", C.c_double), ("joint_nu", C.c_double), ("joint_kt", C.c_double), ("joint_radius", C.c_double),
        ("joint_angle_deg", C.c_double * 16),
        ("muscle_on", C.c_int32), ("reserved2", C.c_int32),
        ("muscle_period", C.c_double), ("muscle_ramp_up_time", C.c_double), ("muscle_phase_shift", C.c_double),
        ("muscle_direction", C.c_double * 3),
        ("spline_dir_mask", C.c_int32), ("spline_n_ctrl", C.c_int32),
        ("spline_scale", C.c_double), ("spline_max_rate", C.c_double),
        ("tip_radius", C.c_double), ("sucker_on", C.c_int32), ("sucker_index", C.c_int32),
        ("taper_node_mean", C.c_int32), ("tm_muscle_on", C.c_int32),
        ("tm_max_stress", C.c_double), ("tm_radius_ref", C.c_double),
        ("muscle_layers_on", C.c_int32), ("head_fixed", C.c_int32),
        ("lm_max_stress", C.c_double), ("lm_px", C.c_double * 2), ("lm_py", C.c_double * 2),
        ("n_fixed_sucker", C.c_int32), ("fixed_sucker_index", C.c_int32 * 3),
    ]


class SrStateView(C.Structure):
    _fields_ = [
        ("base", C.c_void_p), ("n_env", C.c_int32), ("n_fields", C.c_int32), ("stride", C.c_int32),
        ("elem_size", C.c_int32), ("f_position", C.c_int32), ("f_velocity", C.c_int32),
        ("f_director", C.c_int32), ("f_omega", C.c_int32), ("f_tangents", C.c_int32),
        ("f_kappa", C.c_int32), ("f_sigma", C.c_int32), ("f_dilatation", C.c_int32),
    ]


class SoftRodError(RuntimeError):
    pass


_lib = None


def load_library():
    """Load libsoftrod.so (building it with nvcc if the sources are newer)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if _build.is_stale():
        path = _build.build_library()
    if not os.path.exists(path):
        raise SoftRodError(f"{path} missing: build it with `python -m gym_softrobot_b200.build` "
                           "(there is no CPU fallback)")
    L = C.CDLL(path)
    L.sr_abi_version.restype = C.c_int
    L.sr_last_error.restype = C.c_char_p
    L.sr_create.argtypes = [C.POINTER(SrConfig), C.POINTER(C.c_void_p)]
    L.sr_destroy.argtypes = [C.c_void_p]
    L.sr_destroy.restype = None
    for f in ("sr_obs_dim", "sr_action_dim", "sr_init_dim"):
        getattr(L, f).argtypes = [C.c_void_p]
    L.sr_reset.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.sr_step.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.sr_reset_host.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    L.sr_step_host.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    L.sr_observe.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.sr_get_state.argtypes = [C.c_void_p, C.POINTER(SrStateView)]
    L.sr_set_state.argtypes = [C.c_void_p, C.POINTER(SrStateView), C.c_void_p]
    L.sr_copy_from.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.sr_copy_envs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    L.sr_get_aux.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int32)]
    L.sr_get_head.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int32)]
    L.sr_get_rest_kappa.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.sr_get_sucker.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.sr_get_ext_loads.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
    L.sr_get_sucker_index.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.sr_get_tm_activation.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.sr_get_muscle_activation.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.sr_get_fixed_suckers.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.sr_get_muscle.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int32)]
    L.sr_get_spline.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int32)]
    L.sr_spline_basis.argtypes = [C.c_int32, C.c_double, C.c_void_p]
    L.sr_launch_count.argtypes = [C.c_void_p]
    L.sr_launch_count.restype = C.c_int64
    L.sr_fallback_count.argtypes = [C.c_void_p]
    L.sr_fallback_count.restype = C.c_int64
    L.sr_fallback_causes.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
    L.sr_nonplanar_count.argtypes = [C.c_void_p]
    L.sr_nonplanar_count.restype = C.c_int64
    L.sr_measure_fp64_peak.argtypes = [C.c_int, C.POINTER(C.c_double)]
    L.sr_measure_fp64_peak_regs.argtypes = [C.c_int, C.POINTER(C.c_double)]
    L.sr_selftest_reciprocals.argtypes = [C.c_int, C.c_int32, C.c_double, C.c_double, C.POINTER(C.c_double)]
    if L.sr_abi_version() != 1:
        raise SoftRodError("libsoftrod.so ABI version mismatch")
    _lib = L
    return L


def _check(rc):
    if rc != SR_OK:
        raise SoftRodError(f"softrod error {rc}: {load_library().sr_last_error().decode()}")


class _DevMem:
    """Zero-copy torch view of library-owned device memory via __cuda_array_interface__."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {
            "shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2,
            "strides": None,
        }


def copy_env_indices(dst_idx, src_idx, n_dst, n_src):
    """The index pairs of a copy_envs call as two int64 NumPy arrays, checked: ints, sequences, NumPy arrays or torch
    tensors (a CUDA tensor costs one device sync) of integers, equal lengths, every destination in [0, n_dst) and
    every source in [0, n_src), no destination twice.  Raises ValueError otherwise."""
    def as_index(x, what):
        if hasattr(x, "detach"):
            x = x.detach().cpu().numpy()
        a = np.asarray(x)
        if a.ndim == 0:
            a = a.reshape(1)
        if a.ndim != 1:
            raise ValueError(f"{what} must be one-dimensional, got shape {a.shape}")
        if a.size == 0:
            return a.astype(np.int64)
        if a.dtype == np.bool_ or not np.issubdtype(a.dtype, np.integer):
            raise ValueError(f"{what} must hold integers, got {a.dtype}")
        return a.astype(np.int64)
    d, s = as_index(dst_idx, "dst_idx"), as_index(src_idx, "src_idx")
    if d.size != s.size:
        raise ValueError(f"dst_idx and src_idx differ in length ({d.size} and {s.size})")
    if d.size and (d.min() < 0 or d.max() >= n_dst):
        raise ValueError(f"dst_idx out of range [0, {n_dst})")
    if s.size and (s.min() < 0 or s.max() >= n_src):
        raise ValueError(f"src_idx out of range [0, {n_src})")
    if np.unique(d).size != d.size:
        raise ValueError("dst_idx names an env twice")
    return d, s


def spline_basis(n_ctrl: int, base_length: float):
    """Cardinal polynomials [n_ctrl + 1 intervals, n_ctrl, 4] of the not-a-knot cubic the kernel uses
    (sr_spline_basis; host-only, works without a GPU)."""
    import numpy as np
    lib = load_library()
    out = np.zeros((n_ctrl + 1, n_ctrl, 4))
    _check(lib.sr_spline_basis(n_ctrl, float(base_length), out.ctypes.data_as(C.c_void_p)))
    return out


def selftest_reciprocals(n=1 << 20, lo=1e-12, hi=1e12, device=0):
    """(max rel err of rsqrt_nr, of rcp_nr) over n log-spaced arguments (sr_selftest_reciprocals)."""
    lib = load_library()
    out = (C.c_double * 2)()
    _check(lib.sr_selftest_reciprocals(device, n, lo, hi, out))
    return out[0], out[1]


def probe_latency(device=0):
    """dict of dependent-issue latencies in cycles (sr_probe_latency)."""
    lib = load_library()
    lib.sr_probe_latency.argtypes = [C.c_int, C.POINTER(C.c_double)]
    out = (C.c_double * 8)()
    _check(lib.sr_probe_latency(device, out))
    return {"dfma": out[0], "dadd": out[1], "mufu_rsq64h+dfma": out[2], "sts_bar_lds_bar": out[3], "dfma_imm": out[4]}


def measure_fp64_peak(device: int = 0, three_register_operands: bool = False) -> float:
    """DFMA issue peak in TFLOP/s (8 independent chains per thread).  With `three_register_operands` every
    DFMA reads three distinct 64-bit registers, which B200's register file sustains at only 2/3 of the rate."""
    out = C.c_double()
    lib = load_library()
    fn = lib.sr_measure_fp64_peak_regs if three_register_operands else lib.sr_measure_fp64_peak
    _check(fn(device, C.byref(out)))
    return out.value


class Handle:
    """One batched rod simulation on one GPU (wraps sr_handle*)."""

    def __init__(self, *, model, n_env, n_elem, dt, base_length, base_radius, density, youngs_modulus,
                 shear_modulus=0.0, gravity=(0.0, 0.0, 0.0), damping_constant=-1.0, bc_kind=BC_FREE,
                 point_force_on_base=False, damping_before_constraints=False, laplace_filter_order=0,
                 device=0, dtype=DTYPE_F64, math=MATH_FAST, base_step=0.0, base_limit=0.0,
                 base_move_period=0.0, contact=None, n_rod=1, head=None, joint=None, muscle=None, spline=None,
                 tip_radius=0.0, sucker_index=None, taper_node_mean=False, tm_muscle=None,
                 muscle_layers=None, head_fixed=False, fixed_suckers=None):
        self._lib = load_library()
        cfg = SrConfig()
        cfg.struct_size = C.sizeof(SrConfig)
        cfg.device, cfg.model, cfg.dtype, cfg.math = device, model, dtype, math
        cfg.n_env, cfg.n_elem, cfg.bc_kind = n_env, n_elem, bc_kind
        cfg.point_force_on_base = int(point_force_on_base)
        cfg.damping_before_constraints = int(damping_before_constraints)
        cfg.laplace_filter_order = laplace_filter_order
        cfg.dt, cfg.base_length, cfg.base_radius = dt, base_length, base_radius
        cfg.density, cfg.youngs_modulus, cfg.shear_modulus = density, youngs_modulus, shear_modulus
        cfg.gravity[:] = [float(g) for g in gravity]
        cfg.damping_constant = damping_constant
        cfg.base_step, cfg.base_limit, cfg.base_move_period = base_step, base_limit, base_move_period
        if contact is not None:   # plane_origin, plane_normal, k, nu, slip_velocity_tol, static_mu, kinetic_mu
            cfg.contact_on = 1
            cfg.contact_before_forcing = int(contact.get("before_forcing", False))
            cfg.plane_origin[:] = [float(v) for v in contact["plane_origin"]]
            cfg.plane_normal[:] = [float(v) for v in contact["plane_normal"]]
            cfg.contact_k, cfg.contact_nu = contact["k"], contact["nu"]
            cfg.slip_velocity_tol = contact["slip_velocity_tol"]
            cfg.surface_tol = contact.get("surface_tol", 1e-4)   # PyElastica's fixed surface_tol
            cfg.static_mu[:] = [float(v) for v in contact["static_mu"]]
            cfg.kinetic_mu[:] = [float(v) for v in contact["kinetic_mu"]]
        cfg.n_rod_per_env = n_rod
        if head is not None:      # dict: length, radius, density
            cfg.has_head = 1
            cfg.head_length, cfg.head_radius, cfg.head_density = head["length"], head["radius"], head["density"]
        if joint is not None:     # dict: k, nu, kt, radius, angles_deg (one per rod)
            cfg.joint_k, cfg.joint_nu, cfg.joint_kt, cfg.joint_radius = joint["k"], joint["nu"], joint["kt"], joint["radius"]
            for a, ang in enumerate(joint["angles_deg"]):
                cfg.joint_angle_deg[a] = float(ang)
        if muscle is not None:    # dict: period, ramp_up_time, phase_shift, direction (MuscleTorques kwargs)
            cfg.muscle_on = 1
            cfg.muscle_period, cfg.muscle_ramp_up_time = muscle["period"], muscle["ramp_up_time"]
            cfg.muscle_phase_shift = muscle.get("phase_shift", 0.0)
            cfg.muscle_direction[:] = [float(v) for v in muscle["direction"]]
        if spline is not None:    # dict: directions (subset of 0,1,2), n_ctrl, scale, max_rate
            cfg.spline_dir_mask = sum(1 << int(d) for d in spline["directions"])
            cfg.spline_n_ctrl = spline["n_ctrl"]
            cfg.spline_scale, cfg.spline_max_rate = spline["scale"], spline.get("max_rate", float("inf"))
        cfg.tip_radius = float(tip_radius)
        if sucker_index is not None:
            cfg.sucker_on, cfg.sucker_index = 1, int(sucker_index)
        cfg.taper_node_mean = int(taper_node_mean)
        if tm_muscle is not None:   # dict: max_stress, radius_ref (TransverseMuscle of create_es_muscle_layers)
            cfg.tm_muscle_on = 1
            cfg.tm_max_stress, cfg.tm_radius_ref = float(tm_muscle["max_stress"]), float(tm_muscle["radius_ref"])
        if muscle_layers is not None:   # dict: lm_max_stress, lm_positions [(px, py), (px, py)] in units of the radius
            cfg.muscle_layers_on = 1
            cfg.lm_max_stress = float(muscle_layers["lm_max_stress"])
            for m, (px, py) in enumerate(muscle_layers["lm_positions"]):
                cfg.lm_px[m], cfg.lm_py[m] = float(px), float(py)
        cfg.head_fixed = int(head_fixed)
        if fixed_suckers is not None:   # up to three node / element indices, one ControllableFixConstraint each
            cfg.n_fixed_sucker = len(fixed_suckers)
            for s_, loc in enumerate(fixed_suckers):
                cfg.fixed_sucker_index[s_] = int(loc)
        self.n_rod = max(1, n_rod)
        self.cfg = cfg
        self._h = C.c_void_p()
        _check(self._lib.sr_create(C.byref(cfg), C.byref(self._h)))
        self.n_env, self.n_elem, self.device = n_env, n_elem, device
        self.obs_dim = self._lib.sr_obs_dim(self._h)
        self.action_dim = self._lib.sr_action_dim(self._h)
        self._state_tensor = None

    # -- lifetime -----------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.sr_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launch_count(self) -> int:
        return int(self._lib.sr_launch_count(self._h))

    def fallback_count(self) -> int:
        """env-steps the fast-only kernels handed to the safe kernel so far (sr_fallback_count; synchronises)."""
        return int(self._lib.sr_fallback_count(self._h))

    def fallback_causes(self):
        """(rotation, bend, stretch) counts behind fallback_count(), lean kernels only (sr_fallback_causes)."""
        out = (C.c_int64 * 3)()
        _check(self._lib.sr_fallback_causes(self._h, out))
        return tuple(int(v) for v in out)

    def nonplanar_count(self) -> int:
        """env-steps the planar kernel handed to the 3D safe kernel for not being planar (sr_nonplanar_count; synchronises)."""
        return int(self._lib.sr_nonplanar_count(self._h))

    # -- device-pointer entry points (torch tensors on self.device) -----------
    @staticmethod
    def _stream_ptr():
        import torch
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def reset(self, init, env_idx=None):
        """init: float64 cuda tensor [n, 9]; env_idx: int32 cuda tensor [n] or None."""
        n = init.shape[0]
        assert init.is_cuda and init.dtype.itemsize == 8 and init.is_contiguous()
        assert init.shape[1] == self._lib.sr_init_dim(self._h)
        idx_ptr = None
        if env_idx is not None:
            assert env_idx.is_cuda and env_idx.is_contiguous() and env_idx.numel() == n
            idx_ptr = C.c_void_p(env_idx.data_ptr())
        _check(self._lib.sr_reset(self._h, idx_ptr, n, C.c_void_p(init.data_ptr()), self._stream_ptr()))

    def step(self, action, n_substeps, obs, reward, terminated):
        a_ptr = None
        if self.action_dim > 0:
            assert action.is_cuda and action.is_contiguous() and action.numel() == self.n_env * self.action_dim
            a_ptr = C.c_void_p(action.data_ptr())
        _check(self._lib.sr_step(self._h, a_ptr, int(n_substeps), C.c_void_p(obs.data_ptr()),
                                 C.c_void_p(reward.data_ptr()), C.c_void_p(terminated.data_ptr()),
                                 self._stream_ptr()))

    def observe(self, prev_action, obs):
        p = None if prev_action is None else C.c_void_p(prev_action.data_ptr())
        _check(self._lib.sr_observe(self._h, p, C.c_void_p(obs.data_ptr()), self._stream_ptr()))

    # -- host-buffer entry points (NumPy) ---------------------------------------
    def reset_host(self, init, env_idx=None):
        init = np.ascontiguousarray(init, dtype=np.float64)
        n = init.shape[0]
        idx = None
        if env_idx is not None:
            idx = np.ascontiguousarray(env_idx, dtype=np.int32)
            assert idx.size == n
        _check(self._lib.sr_reset_host(self._h, None if idx is None else idx.ctypes.data, n, init.ctypes.data))

    def step_host(self, action, n_substeps, obs=None, reward=None, terminated=None):
        if obs is None:
            obs = np.empty((self.n_env, self.obs_dim), dtype=np.float32)
            reward = np.empty(self.n_env, dtype=np.float64)
            terminated = np.empty(self.n_env, dtype=np.uint8)
        a_ptr = None
        if self.action_dim > 0:
            action = np.ascontiguousarray(action, dtype=np.float32)
            assert action.size == self.n_env * self.action_dim
            a_ptr = action.ctypes.data
        _check(self._lib.sr_step_host(self._h, a_ptr, int(n_substeps), obs.ctypes.data, reward.ctypes.data,
                                      terminated.ctypes.data))
        return obs, reward, terminated

    # -- state views -----------------------------------------------------------
    def state_view(self) -> SrStateView:
        v = SrStateView()
        _check(self._lib.sr_get_state(self._h, C.byref(v)))
        return v

    def state_tensor(self):
        """torch view [n_env, n_fields, stride] (float64 / float32 per dtype) of the live SoA state."""
        import torch
        if self._state_tensor is None:
            v = self.state_view()
            mem = _DevMem(v.base, (v.n_env, v.n_fields, v.stride), "<f8" if v.elem_size == 8 else "<f4")
            self._state_tensor = torch.as_tensor(mem, device=f"cuda:{self.device}")
            self._view = v
        return self._state_tensor

    def fields(self):
        """Reference-named views (SURVEY §8b): [n_env, 3, n+1] / [n_env, 3, 3, n] / [n_env, 3, n];
        multi-rod handles insert a rod axis: [n_env, n_rod, 3, n+1] ..."""
        st = self.state_tensor()
        if self.n_rod > 1:
            out = self._fields_flat(st)
            return {k: v.unflatten(0, (self.n_env, self.n_rod)) for k, v in out.items()}
        return self._fields_flat(st)

    def _fields_flat(self, st):
        v, n = self._view, self.n_elem
        return {
            "position_collection": st[:, v.f_position:v.f_position + 3, :n + 1],
            "velocity_collection": st[:, v.f_velocity:v.f_velocity + 3, :n + 1],
            "director_collection": st[:, v.f_director:v.f_director + 9, :n].unflatten(1, (3, 3)),
            "omega_collection": st[:, v.f_omega:v.f_omega + 3, :n],
            "tangents": st[:, v.f_tangents:v.f_tangents + 3, :n],
            "kappa": st[:, v.f_kappa:v.f_kappa + 3, :n - 1],
            "sigma": st[:, v.f_sigma:v.f_sigma + 3, :n],
            "dilatation": st[:, v.f_dilatation, :n],
        }

    def aux_tensor(self):
        """torch view [n_env, aux_dim] (float64) of the per-env model scratch (sr_get_aux)."""
        import torch
        ptr, dim = C.c_void_p(), C.c_int32()
        _check(self._lib.sr_get_aux(self._h, C.byref(ptr), C.byref(dim)))
        ts = "<f8" if self.cfg.dtype == DTYPE_F64 else "<f4"
        return torch.as_tensor(_DevMem(ptr.value, (self.n_env, dim.value), ts), device=f"cuda:{self.device}")

    def head_tensor(self):
        """torch view [n_env, 20] of the rigid head: x(3) v(3) Q(9, rows) w(3) pinned z (sr_get_head)."""
        import torch
        ptr, dim = C.c_void_p(), C.c_int32()
        _check(self._lib.sr_get_head(self._h, C.byref(ptr), C.byref(dim)))
        ts = "<f8" if self.cfg.dtype == DTYPE_F64 else "<f4"
        return torch.as_tensor(_DevMem(ptr.value, (self.n_env, dim.value), ts), device=f"cuda:{self.device}")

    def rest_kappa_tensor(self):
        """torch view [n_env (* n_rod), 3, n_elem-1] of the per-rod rest curvature (sr_get_rest_kappa)."""
        import torch
        ptr = C.c_void_p()
        _check(self._lib.sr_get_rest_kappa(self._h, C.byref(ptr)))
        v = self.state_view()
        ts = "<f8" if self.cfg.dtype == DTYPE_F64 else "<f4"
        t = torch.as_tensor(_DevMem(ptr.value, (self.n_env * self.n_rod, 3, v.stride), ts),
                            device=f"cuda:{self.device}")
        return t[:, :, :self.n_elem - 1]

    def sucker_tensor(self):
        """torch view [n_env * n_rod] of the ControllableFixConstraint reduction ratios (sr_get_sucker)."""
        import torch
        ptr = C.c_void_p()
        _check(self._lib.sr_get_sucker(self._h, C.byref(ptr)))
        ts = "<f8" if self.cfg.dtype == DTYPE_F64 else "<f4"
        return torch.as_tensor(_DevMem(ptr.value, (self.n_env * self.n_rod,), ts), device=f"cuda:{self.device}")

    def sucker_index_tensor(self):
        """torch view [n_env * n_rod] (int32) of the index each ControllableFixConstraint acts on (sr_get_sucker_index)."""
        import torch
        ptr = C.c_void_p()
        _check(self._lib.sr_get_sucker_index(self._h, C.byref(ptr)))
        return torch.as_tensor(_DevMem(ptr.value, (self.n_env * self.n_rod,), "<i4"), device=f"cuda:{self.device}")

    def tm_activation_tensor(self):
        """torch view [n_env * n_rod] of the transverse-muscle activations (sr_get_tm_activation)."""
        import torch
        ptr = C.c_void_p()
        _check(self._lib.sr_get_tm_activation(self._h, C.byref(ptr)))
        ts = "<f8" if self.cfg.dtype == DTYPE_F64 else "<f4"
        return torch.as_tensor(_DevMem(ptr.value, (self.n_env * self.n_rod,), ts), device=f"cuda:{self.device}")

    def muscle_activation_tensor(self):
        """torch view [n_env * n_rod, 3, n_elem] (float64) of the per-element activations of the muscle layers:
        longitudinal 1, longitudinal 2, transverse (sr_get_muscle_activation)."""
        import torch
        ptr = C.c_void_p()
        _check(self._lib.sr_get_muscle_activation(self._h, C.byref(ptr)))
        return torch.as_tensor(_DevMem(ptr.value, (self.n_env * self.n_rod, 3, self.n_elem), "<f8"), device=f"cuda:{self.device}")

    def fixed_sucker_tensor(self):
        """torch view [n_env * n_rod, 3] (float64) of the fixed-index ControllableFixConstraint ratios (sr_get_fixed_suckers)."""
        import torch
        ptr = C.c_void_p()
        _check(self._lib.sr_get_fixed_suckers(self._h, C.byref(ptr)))
        return torch.as_tensor(_DevMem(ptr.value, (self.n_env * self.n_rod, 3), "<f8"), device=f"cuda:{self.device}")

    def ext_load_tensors(self):
        """(force, couple): torch views [n_env * n_rod, 3, n_elem + 1] / [.., 3, n_elem] of the external nodal forces
        (lab frame) and element couples (material frame) added every substep (sr_get_ext_loads)."""
        import torch
        pf, pc = C.c_void_p(), C.c_void_p()
        _check(self._lib.sr_get_ext_loads(self._h, C.byref(pf), C.byref(pc)))
        v = self.state_view()
        ts = "<f8" if self.cfg.dtype == DTYPE_F64 else "<f4"
        mk = lambda p: torch.as_tensor(_DevMem(p.value, (self.n_env * self.n_rod, 3, v.stride), ts), device=f"cuda:{self.device}")
        return mk(pf)[:, :, :self.n_elem + 1], mk(pc)[:, :, :self.n_elem]

    def muscle_tensor(self):
        """torch view [n_env, n_elem + 2] (float64): simulation time, wave number, beta(s_k) (sr_get_muscle)."""
        import torch
        ptr, dim = C.c_void_p(), C.c_int32()
        _check(self._lib.sr_get_muscle(self._h, C.byref(ptr), C.byref(dim)))
        return torch.as_tensor(_DevMem(ptr.value, (self.n_env, dim.value), "<f8"), device=f"cuda:{self.device}")

    def spline_tensors(self):
        """(points, magnitudes): torch views of the spline-torque state (sr_get_spline), float64:
        points [n_env, 3, 2P+2] = per material direction P targets, P cached values, initial-call flag, pad;
        magnitudes [n_env, 3, n_elem] = the cached per-element torque."""
        import torch
        ptr, dim = C.c_void_p(), C.c_int32()
        _check(self._lib.sr_get_spline(self._h, C.byref(ptr), C.byref(dim)))
        t = torch.as_tensor(_DevMem(ptr.value, (self.n_env, dim.value), "<f8"), device=f"cuda:{self.device}")
        ch = 2 * self.cfg.spline_n_ctrl + 2
        return t[:, :3 * ch].unflatten(1, (3, ch)), t[:, 3 * ch:].unflatten(1, (3, self.n_elem))

    def set_state_from(self, other: "Handle"):
        """Rod arrays only (sr_set_state): see clone_from for a whole-handle copy."""
        v = other.state_view()
        _check(self._lib.sr_set_state(self._h, C.byref(v), self._stream_ptr()))

    def copy_envs(self, dst_idx, src_idx, src: "Handle" = None):
        """Fork envs (sr_copy_envs): env dst_idx[i] of this handle takes everything that evolves or parametrises env
        src_idx[i] of `src` (default: this handle), the per-env rows of what clone_from copies.  Indices: ints,
        sequences, NumPy arrays or torch tensors, checked by copy_env_indices (ValueError).  Stream-ordered on the
        current stream."""
        import torch
        src = self if src is None else src
        d, s = copy_env_indices(dst_idx, src_idx, self.n_env, src.n_env)
        dev = f"cuda:{self.device}"
        dt = torch.as_tensor(d.astype(np.int32), device=dev).contiguous()
        st = torch.as_tensor(s.astype(np.int32), device=dev).contiguous()
        _check(self._lib.sr_copy_envs(self._h, C.c_void_p(dt.data_ptr()), src._h, C.c_void_p(st.data_ptr()),
                                      int(d.size), self._stream_ptr()))

    def clone_from(self, other: "Handle"):
        """Everything that evolves or parametrises the envs (sr_copy_from): rod arrays, BC anchors, base controller,
        rigid heads, rest curvatures, forcing state."""
        _check(self._lib.sr_copy_from(self._h, other._h, self._stream_ptr()))
