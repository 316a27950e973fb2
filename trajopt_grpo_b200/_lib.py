"""ctypes binding of the C ABI in include/trajopt_grpo.h.

The library is the product: if it is missing, or no sm_100 device is present,
every compute entry point raises -- there is NO CPU fallback in this package.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libtrajopt_grpo_b200.so")

TG_MAX_LAYERS = 8
ENV_CARTPOLE, ENV_PENDULUM, ENV_QUADPOLE2D, ENV_QUADPOLE = 0, 1, 2, 3
ACT_IDS = {"ReLU": 0, "Tanh": 1, "Sigmoid": 2}
ACT_PER_LAYER = -1
ABI_VERSION = 2
PREC_F32, PREC_F64 = 0, 1
ADV_GRPO, ADV_PPO_MC, ADV_PPO_GAE = 0, 1, 2


class EnvCfg(C.Structure):
    _fields_ = [("kind", C.c_int32), ("max_steps", C.c_int32), ("dt", C.c_double),
                ("time_limit_step", C.c_int32), ("balanced_limit", C.c_int32), ("phys", C.c_double * 4)]


class MlpCfg(C.Structure):
    _fields_ = [("n_layers", C.c_int32), ("dims", C.c_int32 * (TG_MAX_LAYERS + 1)), ("activation", C.c_int32),
                ("layer_activation", C.c_int32 * TG_MAX_LAYERS)]


class EngineError(RuntimeError):
    pass


_lib = None
_lock = threading.Lock()
_ctxs: dict[int, C.c_void_p] = {}

_vp, _i64, _i32, _u64, _f, _d = C.c_void_p, C.c_int64, C.c_int, C.c_uint64, C.c_float, C.c_double
_SIGS = {
    "tg_abi_version": (C.c_int, []),
    "tg_last_error": (C.c_char_p, []),
    "tg_ctx_create": (C.c_int, [_i32, C.POINTER(_vp)]),
    "tg_ctx_destroy": (None, [_vp]),
    "tg_ctx_sm_count": (C.c_int, [_vp]),
    "tg_ctx_set_math": (C.c_int, [_vp, _i32]),
    "tg_fp32_peak": (C.c_int, [_vp, C.POINTER(C.c_double)]),
    "tg_tmem_probe": (C.c_int, [_vp, _i32, C.POINTER(C.c_longlong)]),
    "tg_umma_selftest": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp]),
    "tg_env_dims": (C.c_int, [_i32, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "tg_mlp_param_count": (_i64, [C.POINTER(MlpCfg)]),
    "tg_rollout": (C.c_int, [_vp, C.POINTER(EnvCfg), C.POINTER(MlpCfg), _i32, _i64, _vp, _vp, C.POINTER(_f), _vp,
                             _u64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tg_noise_fill": (C.c_int, [_vp, _u64, _i64, _i64, _i32, _i32, _vp, _vp]),
    "tg_env_step": (C.c_int, [_vp, C.POINTER(EnvCfg), _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tg_env_dynamics": (C.c_int, [_vp, C.POINTER(EnvCfg), _i32, _i64, _vp, _vp, _vp, _vp]),
    "tg_quadrotor12_dynamics": (C.c_int, [_vp, _i32, _i64, _d, _vp, _vp, _vp, _vp]),
    "tg_policy_forward": (C.c_int, [_vp, C.POINTER(MlpCfg), _i64, _vp, _vp, C.POINTER(_f), _vp, _vp, _vp, _vp]),
    "tg_policy_forward_traj": (C.c_int, [_vp, C.POINTER(MlpCfg), _i64, _i32, _vp, _vp, _vp, _vp, C.POINTER(_f), _vp,
                                         _vp, _vp]),
    "tg_advantage_workspace_bytes": (_i64, [_i64, _i32]),
    "tg_advantage": (C.c_int, [_vp, _i32, _i64, _i32, _i32, _d, _d, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tg_advantage_ppo_raw": (C.c_int, [_vp, _i32, _i64, _i32, _i32, _d, _d, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tg_advantage_ppo_normalize": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp]),
    "tg_export_trajectory": (C.c_int, [_vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tg_policy_grad_workspace_bytes": (_i64, [_vp, C.POINTER(MlpCfg)]),
    "tg_len_order_hold": (C.c_int, [_vp, _i64, _i32, _vp, _vp]),
    "tg_len_order_release": (C.c_int, [_vp]),
    "tg_policy_grad_scratch_bytes": (C.c_int, [_vp, C.POINTER(MlpCfg), _i64, C.POINTER(_i64), C.POINTER(_i64)]),
    "tg_policy_grad": (C.c_int, [_vp, C.POINTER(MlpCfg), _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(_f),
                                 _f, _f, _f, _vp, _vp, _vp, _vp]),
    "tg_policy_grad_ref": (C.c_int, [_vp, C.POINTER(MlpCfg), _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                     C.POINTER(_f), _f, _f, _f, _f, _vp, _vp, _vp, _vp]),
    "tg_value_grad": (C.c_int, [_vp, C.POINTER(MlpCfg), _i64, _i32, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp, _vp]),
    "tg_policy_grad_batch": (C.c_int, [_vp, C.POINTER(MlpCfg), _i64, _i32, _vp, _vp, _vp, _vp, _vp, _i64, _vp,
                                       C.POINTER(_f), _f, _f, _f, _vp, _vp, _vp, _vp]),
    "tg_value_grad_batch": (C.c_int, [_vp, C.POINTER(MlpCfg), _i64, _i32, _vp, _vp, _vp, _i64, _vp, _f, _vp, _vp, _vp,
                                      _vp]),
    "tg_minibatch_plan_workspace_bytes": (_i64, [_i64]),
    "tg_minibatch_plan": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _vp]),
    "tg_adam_step": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _i64, _d, _d, _d, _d, _vp]),
    "tg_comm_handle_bytes": (C.c_int, []),
    "tg_comm_create": (C.c_int, [_vp, _i32, _i32, _i64, C.POINTER(_vp), _vp]),
    "tg_comm_connect": (C.c_int, [_vp, _vp]),
    "tg_comm_destroy": (C.c_int, [_vp]),
    "tg_comm_grad_slot": (C.c_int, [_vp, C.POINTER(_vp)]),
    "tg_allreduce_adam_step": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _i64, _d, _d, _d, _d, _vp, _vp]),
}
EXPORTS = tuple(_SIGS)


def load():
    """dlopen the in-tree library and attach signatures (no device needed)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise EngineError(
                    f"{LIB_PATH} is missing: build it with `python -m trajopt_grpo_b200._build` "
                    "(there is no CPU fallback)")
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in _SIGS.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            if lib.tg_abi_version() != ABI_VERSION:
                raise EngineError(f"{LIB_PATH} has ABI version {lib.tg_abi_version()}, this package binds "
                                  f"version {ABI_VERSION}: rebuild with `python -m trajopt_grpo_b200._build --force`")
            _lib = lib
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().tg_last_error().decode(errors="replace")
        raise EngineError(f"{what} failed (status {rc}): {msg}")


def ctx(device=None) -> C.c_void_p:
    """One engine context per CUDA device (lazily created)."""
    lib = load()
    if not torch.cuda.is_available():
        raise EngineError("no CUDA device: the trajopt_grpo_b200 engine has no CPU fallback")
    idx = torch.cuda.current_device() if device is None else torch.device(device).index
    if idx is None:
        idx = torch.cuda.current_device()
    with _lock:
        if idx not in _ctxs:
            h = _vp()
            check(lib.tg_ctx_create(idx, C.byref(h)), "tg_ctx_create")
            _ctxs[idx] = h
    return _ctxs[idx]


def is_checkpoint_writer() -> bool:
    """In a sharded run (torch.distributed initialised) every rank holds the same weights, optimizer state and reward
    history, and the reference's Pipeline.save would make each of them write the same files: only rank 0 writes."""
    import torch.distributed as dist
    return not (dist.is_available() and dist.is_initialized()) or dist.get_rank() == 0


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t):
    return None if t is None else t.data_ptr()


def mlp_cfg(dims, activation="ReLU") -> MlpCfg:
    dims = [int(d) for d in dims]
    if len(dims) - 1 > TG_MAX_LAYERS or len(dims) < 2:
        raise EngineError(f"MLP with {len(dims) - 1} Linear layers is outside [1, {TG_MAX_LAYERS}]")
    # models/neural_network.py:38-45: one torch.nn class name for every hidden layer, or a list with one per layer
    names = list(activation) if isinstance(activation, (list, tuple)) else [activation] * max(len(dims) - 2, 1)
    if isinstance(activation, (list, tuple)) and len(names) != len(dims) - 2:
        raise EngineError("Number of activation functions must equal the number of hidden layers.")
    for nm in names:
        if nm not in ACT_IDS:
            raise EngineError(f"activation {nm!r} is not supported by the kernels ({sorted(ACT_IDS)})")
    cfg = MlpCfg()
    cfg.n_layers = len(dims) - 1
    for i, d in enumerate(dims):
        cfg.dims[i] = d
    if len(set(names)) <= 1:
        cfg.activation = ACT_IDS[names[0]] if names else 0
    else:
        cfg.activation = ACT_PER_LAYER          # FP32-pipe kernels; the tensor-core kernels take one activation
        for i, nm in enumerate(names):
            cfg.layer_activation[i] = ACT_IDS[nm]
    return cfg


def time_limit_step(dt: float, max_steps: int) -> int:
    """First step count at which the reference's float64 `_time > max_time` fires
    (cartpole_env.py:153,168; pendulum_env.py:137,154): replay the accumulation."""
    max_time = max_steps * dt
    t = 0
    for k in range(1, max_steps + 3):
        t += dt
        if t > max_time:
            return k
    return max_steps + 3


def balanced_limit_count(dt: float, limit: float = 5.0) -> int:
    """Consecutive balanced steps at which float64 `_time_balanced > 5` fires
    (pendulum_env.py:138,155)."""
    tb, c = 0, 0
    while True:
        tb = tb + dt
        c += 1
        if tb > limit:
            return c
        if c > 10_000_000:
            raise EngineError("timestep too small for the balanced-time threshold")


def env_cfg(kind: int, max_steps: int, dt: float, phys=None) -> EnvCfg:
    """`phys`: the env's physical constructor arguments (CartPole: masscart, masspole, length, gravity;
    Pendulum: mass, length, gravity); None = the reference's defaults."""
    cfg = EnvCfg()
    cfg.kind, cfg.max_steps, cfg.dt = int(kind), int(max_steps), float(dt)
    for i, v in enumerate(phys or ()):
        cfg.phys[i] = float(v)
    cfg.time_limit_step = time_limit_step(float(dt), int(max_steps)) if kind in (ENV_CARTPOLE, ENV_PENDULUM) else 0
    cfg.balanced_limit = balanced_limit_count(float(dt)) if kind == ENV_PENDULUM else 0
    return cfg


def cov_array(cov_diag):
    arr = (C.c_float * len(cov_diag))(*[float(c) for c in cov_diag])
    return arr
