"""Tensor-level wrappers over the C ABI (include/trajopt_grpo.h).

Every function takes/returns CUDA torch tensors in the kernels' native
struct-of-arrays layout (env / sample index innermost) and launches on torch's
current stream.  PyTorch is plumbing here (device memory and streams); all
arithmetic happens in the sm_100a kernels behind the ABI.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L

OBS_DIM = {L.ENV_CARTPOLE: 5, L.ENV_PENDULUM: 3, L.ENV_QUADPOLE2D: 10, L.ENV_QUADPOLE: 20}
ACT_DIM = {L.ENV_CARTPOLE: 1, L.ENV_PENDULUM: 1, L.ENV_QUADPOLE2D: 2, L.ENV_QUADPOLE: 4}

_ws_cache: dict = {}

# kernels of THIS library launched through the wrappers (bench.py reports it as gpu_launches)
COUNTERS = {"launches": 0}


def _count(n: int):
    COUNTERS["launches"] += n


MATH_AUTO, MATH_FP32, MATH_3XTF32 = 0, 1, 2
_MATH_NAMES = {"auto": MATH_AUTO, "fp32": MATH_FP32, "3xtf32": MATH_3XTF32}


def set_math(mode, device=None):
    """tg_ctx_set_math: 'auto' (tensor cores when the policy shape is eligible), 'fp32', '3xtf32'."""
    lib = L.load()
    m = _MATH_NAMES[mode] if isinstance(mode, str) else int(mode)
    L.check(lib.tg_ctx_set_math(L.ctx(device), m), "tg_ctx_set_math")


def fp32_peak_tflops(device=None) -> float:
    """Measured FP32 FMA-pipe throughput (tg_fp32_peak)."""
    lib = L.load()
    out = C.c_double()
    L.check(lib.tg_fp32_peak(L.ctx(device), C.byref(out)), "tg_fp32_peak")
    return float(out.value)


def _need(t: torch.Tensor, dtype, name: str, shape=None):
    if not (isinstance(t, torch.Tensor) and t.is_cuda):
        raise L.EngineError(f"{name} must be a CUDA tensor (no CPU fallback)")
    if t.dtype != dtype:
        raise L.EngineError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise L.EngineError(f"{name} must be contiguous")
    if shape is not None and tuple(t.shape) != tuple(shape):
        raise L.EngineError(f"{name} has shape {tuple(t.shape)}, expected {tuple(shape)}")
    return t


def _workspace(key, nbytes: int, device) -> torch.Tensor:
    k = (key, torch.device(device).index)
    ws = _ws_cache.get(k)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        _ws_cache[k] = ws
    return ws


def rollout(kind, max_steps, dt, dims, activation, params, cov_diag, init_state, noise=None, seed=0,
            want_logp=True, out=None, env_offset=0, phys=None):
    """tg_rollout.  init_state [S,N] float32 (throughput) or float64 (parity).
    Returns dict(obs [T,O,N], act [T,A,N], rew [T,N], logp [T,N], len [N] i32, ret [N])."""
    lib = L.load()
    O, A = OBS_DIM[kind], ACT_DIM[kind]
    T = int(max_steps)
    if init_state.dtype not in (torch.float32, torch.float64):
        raise L.EngineError("init_state must be float32 or float64")
    _need(init_state, init_state.dtype, "init_state")
    if init_state.shape[0] != O:
        raise L.EngineError(f"init_state must be [S={O}, N]")
    N = init_state.shape[1]
    dev = init_state.device
    _need(params, torch.float32, "params")
    if noise is not None:
        _need(noise, torch.float32, "noise", (T, A, N))
    if out is not None and (tuple(out["obs"].shape) != (T, O, N) or out["obs"].device != dev):
        out = None
    if out is None:
        out = {
            "obs": torch.empty((T, O, N), dtype=torch.float32, device=dev),
            "act": torch.empty((T, A, N), dtype=torch.float32, device=dev),
            "rew": torch.empty((T, N), dtype=torch.float32, device=dev),
            "logp": torch.empty((T, N), dtype=torch.float32, device=dev) if want_logp else None,
            "len": torch.empty((N,), dtype=torch.int32, device=dev),
            "ret": torch.empty((N,), dtype=torch.float32, device=dev),
        }
    ecfg = L.env_cfg(kind, T, dt, phys)
    mcfg = L.mlp_cfg(dims, activation)
    prec = L.PREC_F64 if init_state.dtype == torch.float64 else L.PREC_F32
    with torch.cuda.device(dev):
        rc = lib.tg_rollout(L.ctx(dev), C.byref(ecfg), C.byref(mcfg), prec, N, L.ptr(init_state), L.ptr(params),
                            L.cov_array(cov_diag), L.ptr(noise), int(seed) & (2 ** 64 - 1), int(env_offset),
                            L.ptr(out["obs"]),
                            L.ptr(out["act"]), L.ptr(out["rew"]), L.ptr(out.get("logp")), L.ptr(out["len"]),
                            L.ptr(out.get("ret")), L.stream_ptr())
    L.check(rc, "tg_rollout")
    _count(2)
    return out


def noise_fill(seed, N, T, A, device=None, env_offset=0):
    lib = L.load()
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    out = torch.empty((T, A, N), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        L.check(lib.tg_noise_fill(L.ctx(dev), int(seed) & (2 ** 64 - 1), int(env_offset), N, T, A, L.ptr(out),
                                  L.stream_ptr()),
                "tg_noise_fill")
    _count(1)
    return out


def env_step(kind, max_steps, dt, state, raw_action, steps_done=None, bal_count=None, phys=None):
    """tg_env_step.  state [S,N] f32|f64, raw_action [A,N] f32 -> (next, reward, done i32, bal i32)."""
    lib = L.load()
    O, A = OBS_DIM[kind], ACT_DIM[kind]
    _need(state, state.dtype, "state")
    N = state.shape[1]
    dev = state.device
    _need(raw_action, torch.float32, "raw_action", (A, N))
    if steps_done is not None:
        _need(steps_done, torch.int32, "steps_done", (N,))
    if bal_count is not None:
        _need(bal_count, torch.int32, "bal_count", (N,))
    nxt = torch.empty_like(state)
    rew = torch.empty((N,), dtype=state.dtype, device=dev)
    done = torch.empty((N,), dtype=torch.int32, device=dev)
    bal = torch.empty((N,), dtype=torch.int32, device=dev)
    ecfg = L.env_cfg(kind, max_steps, dt, phys)
    prec = L.PREC_F64 if state.dtype == torch.float64 else L.PREC_F32
    with torch.cuda.device(dev):
        rc = lib.tg_env_step(L.ctx(dev), C.byref(ecfg), prec, N, L.ptr(state), L.ptr(raw_action), L.ptr(steps_done),
                             L.ptr(bal_count), L.ptr(nxt), L.ptr(rew), L.ptr(done), L.ptr(bal), L.stream_ptr())
    L.check(rc, "tg_env_step")
    _count(1)
    return nxt, rew, done, bal


def env_dynamics(kind, dt, state, control, phys=None):
    """tg_env_dynamics: Env._dynamics for N envs.  state [S,N] f32|f64, control [A,N] f32 (already wrapped)
    -> next state [S,N]."""
    lib = L.load()
    O, A = OBS_DIM[kind], ACT_DIM[kind]
    _need(state, state.dtype, "state")
    if state.dtype not in (torch.float32, torch.float64) or state.shape[0] != O:
        raise L.EngineError(f"state must be [S={O}, N] float32 or float64")
    N = state.shape[1]
    _need(control, torch.float32, "control", (A, N))
    nxt = torch.empty_like(state)
    ecfg = L.env_cfg(kind, 1, dt, phys)
    prec = L.PREC_F64 if state.dtype == torch.float64 else L.PREC_F32
    with torch.cuda.device(state.device):
        rc = lib.tg_env_dynamics(L.ctx(state.device), C.byref(ecfg), prec, N, L.ptr(state), L.ptr(control), L.ptr(nxt),
                                 L.stream_ptr())
    L.check(rc, "tg_env_dynamics")
    _count(1)
    return nxt


def quadrotor12_dynamics(state, control, dt=0.05):
    lib = L.load()
    _need(state, state.dtype, "state")
    _need(control, state.dtype, "control", (4, state.shape[1]))
    out = torch.empty_like(state)
    prec = L.PREC_F64 if state.dtype == torch.float64 else L.PREC_F32
    with torch.cuda.device(state.device):
        L.check(lib.tg_quadrotor12_dynamics(L.ctx(state.device), prec, state.shape[1], float(dt), L.ptr(state),
                                            L.ptr(control), L.ptr(out), L.stream_ptr()), "tg_quadrotor12_dynamics")
    _count(1)
    return out


def policy_forward(dims, activation, params, x, cov_diag=None, act=None, want_mu=True, want_logp=False):
    """tg_policy_forward.  x [K0,M] -> (mu [A,M] | None, logp [M] | None)."""
    lib = L.load()
    _need(x, torch.float32, "x")
    M = x.shape[1]
    A = int(dims[-1])
    dev = x.device
    _need(params, torch.float32, "params")
    mu = torch.empty((A, M), dtype=torch.float32, device=dev) if want_mu else None
    logp = torch.empty((M,), dtype=torch.float32, device=dev) if want_logp else None
    if act is not None:
        _need(act, torch.float32, "act", (A, M))
    mcfg = L.mlp_cfg(dims, activation)
    cov = L.cov_array(cov_diag) if cov_diag is not None else None
    with torch.cuda.device(dev):
        rc = lib.tg_policy_forward(L.ctx(dev), C.byref(mcfg), M, L.ptr(x), L.ptr(params), cov, L.ptr(act), L.ptr(mu),
                                   L.ptr(logp), L.stream_ptr())
    L.check(rc, "tg_policy_forward")
    _count(2)
    return mu, logp


def policy_forward_traj(dims, activation, params, obs, cov_diag=None, act=None, length=None, want_mu=False,
                        want_logp=True, out_mu=None, out_logp=None):
    """tg_policy_forward_traj.  obs [T,O,N] (+ act [T,A,N]) -> (mu [T,A,N] | None, logp [T,N] | None);
    rows past `length` are left unwritten: zero in the tensors allocated here, unchanged in `out_mu` / `out_logp`
    (given, they are written in place and imply want_mu / want_logp)."""
    lib = L.load()
    _need(obs, torch.float32, "obs")
    T, O, N = obs.shape
    A = int(dims[-1])
    dev = obs.device
    _need(params, torch.float32, "params")
    if act is not None:
        _need(act, torch.float32, "act", (T, A, N))
    if length is not None:
        _need(length, torch.int32, "len", (N,))
    if out_mu is not None:
        mu = _need(out_mu, torch.float32, "out_mu", (T, A, N))
    else:
        mu = torch.zeros((T, A, N), dtype=torch.float32, device=dev) if want_mu else None
    if out_logp is not None:
        logp = _need(out_logp, torch.float32, "out_logp", (T, N))
    else:
        logp = torch.zeros((T, N), dtype=torch.float32, device=dev) if want_logp else None
    mcfg = L.mlp_cfg(dims, activation)
    cov = L.cov_array(cov_diag) if cov_diag is not None else None
    with torch.cuda.device(dev):
        rc = lib.tg_policy_forward_traj(L.ctx(dev), C.byref(mcfg), N, T, L.ptr(obs), L.ptr(act), L.ptr(length),
                                        L.ptr(params), cov, L.ptr(mu), L.ptr(logp), L.stream_ptr())
    L.check(rc, "tg_policy_forward_traj")
    _count(2 + (2 if length is not None else 0))   # + order_keys / order_count (the radix sort is CUB's)
    return mu, logp


def advantage(mode, G, E, T, gamma, lam, rew, length, values=None, want_rtg=False):
    """tg_advantage.  rew [T,N], length [N] i32 -> (adv [T,N], rtg [T,N] | None)."""
    lib = L.load()
    N = G * E
    _need(rew, torch.float32, "rew", (T, N))
    _need(length, torch.int32, "len", (N,))
    dev = rew.device
    adv = torch.empty_like(rew)
    need_rtg = want_rtg or mode != L.ADV_GRPO
    rtg = torch.empty_like(rew) if need_rtg else None
    if values is not None:
        _need(values, torch.float32, "values", (T, N))
    ws = _workspace("adv", lib.tg_advantage_workspace_bytes(N, G), dev)
    with torch.cuda.device(dev):
        rc = lib.tg_advantage(L.ctx(dev), mode, G, E, T, float(gamma), float(lam), L.ptr(rew), L.ptr(length),
                              L.ptr(values), L.ptr(adv), L.ptr(rtg), L.ptr(ws), L.stream_ptr())
    L.check(rc, "tg_advantage")
    _count(1 if mode == L.ADV_GRPO else 3)
    return adv, rtg


def advantage_ppo_raw(mode, G, E, T, gamma, lam, rew, length, values, out_adv=None, out_rtg=None):
    """tg_advantage_ppo_raw -> (raw adv [T,N], raw returns [T,N], sums [5] float64 =
    (sum adv, sum adv^2, sum ret, sum ret^2, n valid)).  The sums are additive over ranks (and over chunks of whole
    groups).  `out_adv` / `out_rtg`, when given, receive the raw values (every row is written)."""
    lib = L.load()
    N = G * E
    _need(rew, torch.float32, "rew", (T, N))
    _need(length, torch.int32, "len", (N,))
    _need(values, torch.float32, "values", (T, N))
    dev = rew.device
    adv = torch.empty_like(rew) if out_adv is None else _need(out_adv, torch.float32, "out_adv", (T, N))
    rtg = torch.empty_like(rew) if out_rtg is None else _need(out_rtg, torch.float32, "out_rtg", (T, N))
    sums = torch.empty((5,), dtype=torch.float64, device=dev)
    ws = _workspace("adv", lib.tg_advantage_workspace_bytes(N, G), dev)
    with torch.cuda.device(dev):
        rc = lib.tg_advantage_ppo_raw(L.ctx(dev), mode, G, E, T, float(gamma), float(lam), L.ptr(rew), L.ptr(length),
                                      L.ptr(values), L.ptr(adv), L.ptr(rtg), L.ptr(sums), L.ptr(ws), L.stream_ptr())
    L.check(rc, "tg_advantage_ppo_raw")
    _count(2)
    return adv, rtg, sums


def advantage_ppo_normalize(T, length, sums, adv, rtg):
    """tg_advantage_ppo_normalize: z-score adv and rtg in place with the (global) sums."""
    lib = L.load()
    N = length.shape[0]
    _need(adv, torch.float32, "adv", (T, N))
    _need(rtg, torch.float32, "rtg", (T, N))
    _need(sums, torch.float64, "sums", (5,))
    dev = adv.device
    with torch.cuda.device(dev):
        rc = lib.tg_advantage_ppo_normalize(L.ctx(dev), N, T, L.ptr(length), L.ptr(sums), L.ptr(adv), L.ptr(rtg),
                                            L.stream_ptr())
    L.check(rc, "tg_advantage_ppo_normalize")
    _count(1)
    return adv, rtg


def policy_grad(dims, activation, params, cov_diag, obs, act, adv, old_logp, length, eps_clip, scale, kl_scale=0.0,
                out_grad=None, ref_logp=None, ref_scale=0.0):
    """tg_policy_grad -> (grad [n_params], stats [4] = objective, n_valid, sum ratio, n_clipped).

    With `ref_logp` [T,N] (log-probs of `act` under a frozen reference policy): tg_policy_grad_ref, GRPO's k3 KL
    penalty -ref_scale * sum(exp(u) - u - 1), u = ref_logp - logp, added to the objective (ref_scale = beta * scale),
    and stats [5] = objective, n_valid, sum ratio, n_clipped, sum(exp(u) - u - 1)."""
    lib = L.load()
    T, O, N = obs.shape
    A = act.shape[1]
    _need(obs, torch.float32, "obs")
    _need(act, torch.float32, "act", (T, A, N))
    _need(adv, torch.float32, "adv", (T, N))
    _need(old_logp, torch.float32, "old_logp", (T, N))
    _need(length, torch.int32, "len", (N,))
    _need(params, torch.float32, "params")
    if ref_logp is not None:
        _need(ref_logp, torch.float32, "ref_logp", (T, N))
    dev = obs.device
    mcfg = L.mlp_cfg(dims, activation)
    grad = torch.empty_like(params) if out_grad is None else out_grad
    stats = torch.empty((4 if ref_logp is None else 5,), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        ws = _workspace("grad", lib.tg_policy_grad_workspace_bytes(L.ctx(dev), C.byref(mcfg)), dev)
        if ref_logp is None:
            rc = lib.tg_policy_grad(L.ctx(dev), C.byref(mcfg), N, T, L.ptr(obs), L.ptr(act), L.ptr(adv),
                                    L.ptr(old_logp), L.ptr(length), L.ptr(params), L.cov_array(cov_diag),
                                    float(eps_clip), float(scale), float(kl_scale), L.ptr(grad), L.ptr(stats),
                                    L.ptr(ws), L.stream_ptr())
        else:
            rc = lib.tg_policy_grad_ref(L.ctx(dev), C.byref(mcfg), N, T, L.ptr(obs), L.ptr(act), L.ptr(adv),
                                        L.ptr(old_logp), L.ptr(ref_logp), L.ptr(length), L.ptr(params),
                                        L.cov_array(cov_diag), float(eps_clip), float(scale), float(kl_scale),
                                        float(ref_scale), L.ptr(grad), L.ptr(stats), L.ptr(ws), L.stream_ptr())
    L.check(rc, "tg_policy_grad")
    _count(3 if length_order.held else 5)          # pack, [order_keys, order_count,] update, grad_reduce
    return grad, stats


class length_order:
    """with engine.length_order(r.len, T): the length order of the rollout is built once (tg_len_order_hold) and
    reused by every policy_grad / value_grad / policy_forward_traj call inside the block."""
    held = False

    def __init__(self, length, T):
        self.length, self.T = length, int(T)

    def __enter__(self):
        lib = L.load()
        _need(self.length, torch.int32, "len")
        dev = self.length.device
        with torch.cuda.device(dev):
            L.check(lib.tg_len_order_hold(L.ctx(dev), self.length.numel(), self.T, L.ptr(self.length), L.stream_ptr()),
                    "tg_len_order_hold")
        _count(2)
        length_order.held = True
        return self

    def __exit__(self, *exc):
        length_order.held = False
        L.check(L.load().tg_len_order_release(L.ctx(self.length.device)), "tg_len_order_release")
        return False


def policy_grad_traffic_bytes(dims, n_valid: int, length, activation="ReLU"):
    """HBM bytes one tg_policy_grad launch moves for a rollout with episode lengths `length` [N] i32:
    algorithmic trajectory reads (obs + act + adv + old log-prob of every valid step) plus the scratch the
    streamed wide tensor-core path writes and reads back (tg_policy_grad_scratch_bytes)."""
    lib = L.load()
    T_max = int(length.max().item())
    live = (length.view(1, -1) > torch.arange(T_max, device=length.device).view(-1, 1)).sum(1)      # envs alive per step
    n_tiles = int(((live + 127) // 128).sum().item())
    w, r = C.c_int64(), C.c_int64()
    mcfg = L.mlp_cfg(dims, activation)
    L.check(lib.tg_policy_grad_scratch_bytes(L.ctx(length.device), C.byref(mcfg), n_tiles, C.byref(w), C.byref(r)),
            "tg_policy_grad_scratch_bytes")
    alg = 4 * (dims[0] + dims[-1] + 2) * int(n_valid)
    return {"algorithmic_read": alg, "scratch_written": int(w.value), "scratch_read": int(r.value),
            "total": alg + int(w.value) + int(r.value), "live_tiles": n_tiles}


def policy_grad_batch(dims, activation, params, cov_diag, obs, act, adv, old_logp, sample_ids, eps_clip, scale,
                      kl_scale=0.0, out_grad=None):
    """tg_policy_grad_batch: the clipped-surrogate gradient over the samples listed in `sample_ids`
    (int64 flat slot ids t*N + n)."""
    lib = L.load()
    T, O, N = obs.shape
    A = act.shape[1]
    _need(obs, torch.float32, "obs")
    _need(act, torch.float32, "act", (T, A, N))
    _need(adv, torch.float32, "adv", (T, N))
    _need(old_logp, torch.float32, "old_logp", (T, N))
    _need(sample_ids, torch.int64, "sample_ids")
    _need(params, torch.float32, "params")
    dev = obs.device
    mcfg = L.mlp_cfg(dims, activation)
    grad = torch.empty_like(params) if out_grad is None else out_grad
    stats = torch.empty((4,), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        ws = _workspace("grad", lib.tg_policy_grad_workspace_bytes(L.ctx(dev), C.byref(mcfg)), dev)
        rc = lib.tg_policy_grad_batch(L.ctx(dev), C.byref(mcfg), N, T, L.ptr(obs), L.ptr(act), L.ptr(adv),
                                      L.ptr(old_logp), L.ptr(sample_ids), sample_ids.numel(), L.ptr(params),
                                      L.cov_array(cov_diag), float(eps_clip), float(scale), float(kl_scale),
                                      L.ptr(grad), L.ptr(stats), L.ptr(ws), L.stream_ptr())
    L.check(rc, "tg_policy_grad_batch")
    _count(3)
    return grad, stats


def value_grad_batch(dims, activation, params, obs, target, sample_ids, scale, out_grad=None):
    """tg_value_grad_batch: critic MSE gradient over the listed samples."""
    lib = L.load()
    T, O, N = obs.shape
    _need(obs, torch.float32, "obs")
    _need(target, torch.float32, "target", (T, N))
    _need(sample_ids, torch.int64, "sample_ids")
    _need(params, torch.float32, "params")
    dev = obs.device
    mcfg = L.mlp_cfg(dims, activation)
    grad = torch.empty_like(params) if out_grad is None else out_grad
    stats = torch.empty((4,), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        ws = _workspace("grad", lib.tg_policy_grad_workspace_bytes(L.ctx(dev), C.byref(mcfg)), dev)
        rc = lib.tg_value_grad_batch(L.ctx(dev), C.byref(mcfg), N, T, L.ptr(obs), L.ptr(target), L.ptr(sample_ids),
                                     sample_ids.numel(), L.ptr(params), float(scale), L.ptr(grad), L.ptr(stats),
                                     L.ptr(ws), L.stream_ptr())
    L.check(rc, "tg_value_grad_batch")
    _count(3)
    return grad, stats


def value_grad(dims, activation, params, obs, target, length, scale, out_grad=None):
    """tg_value_grad -> (grad [n_params], stats[0] = sum of squared errors, stats[1] = n_valid)."""
    lib = L.load()
    T, O, N = obs.shape
    _need(obs, torch.float32, "obs")
    _need(target, torch.float32, "target", (T, N))
    _need(length, torch.int32, "len", (N,))
    _need(params, torch.float32, "params")
    dev = obs.device
    mcfg = L.mlp_cfg(dims, activation)
    grad = torch.empty_like(params) if out_grad is None else out_grad
    stats = torch.empty((4,), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        ws = _workspace("grad", lib.tg_policy_grad_workspace_bytes(L.ctx(dev), C.byref(mcfg)), dev)
        rc = lib.tg_value_grad(L.ctx(dev), C.byref(mcfg), N, T, L.ptr(obs), L.ptr(target), L.ptr(length),
                               L.ptr(params), float(scale), L.ptr(grad), L.ptr(stats), L.ptr(ws), L.stream_ptr())
    L.check(rc, "tg_value_grad")
    _count(5)
    return grad, stats


def minibatch_plan(perm, length, batch_size, base, n_local=None):
    """tg_minibatch_plan: this shard's part of every minibatch of one PPO epoch.

    perm [n_total] int64 (device): the epoch's permutation of the valid steps of the WHOLE rollout (global env index
    major, step minor); length [N] int32: this shard's episode lengths; base: global index of its first valid step.
    `n_local` (= length.sum()) may be passed when the caller knows it, which saves a device-to-host copy.
    Returns (ids [n_local] int64 device: flat slot ids t*N + n in perm order, offsets [n_batches + 1] int64 host):
    minibatch b of this shard is ids[offsets[b]:offsets[b + 1]].  Raises EngineError unless the plan holds exactly
    n_local entries (perm is not a permutation of range(n_total))."""
    lib = L.load()
    _need(perm, torch.int64, "perm")
    _need(length, torch.int32, "len")
    if perm.dim() != 1 or length.dim() != 1 or perm.numel() == 0 or length.numel() == 0:
        raise L.EngineError("perm and len must be non-empty 1-d tensors")
    if int(batch_size) <= 0:
        raise L.EngineError(f"batch_size must be positive, got {batch_size}")
    dev = perm.device
    n_total, N = perm.numel(), length.numel()
    row0 = torch.cumsum(length.to(torch.int64), 0)
    if n_local is None:
        n_local = int(row0[-1].item())
    row0.sub_(length)
    n_batches = -(-n_total // int(batch_size))
    ids = torch.empty((int(n_local),), dtype=torch.int64, device=dev)
    offsets = torch.empty((n_batches + 1,), dtype=torch.int64, device=dev)
    ws = _workspace("plan", lib.tg_minibatch_plan_workspace_bytes(n_total), dev)
    with torch.cuda.device(dev):
        rc = lib.tg_minibatch_plan(L.ctx(dev), N, L.ptr(length), L.ptr(row0), L.ptr(perm), n_total, int(batch_size),
                                   int(base), int(n_local), ids.numel(), L.ptr(ids), L.ptr(offsets), L.ptr(ws),
                                   L.stream_ptr())
    L.check(rc, "tg_minibatch_plan")
    _count(3)
    offsets = offsets.cpu()
    if int(offsets[-1]) != int(n_local):
        raise L.EngineError(f"tg_minibatch_plan: {int(offsets[-1])} entries of perm fall in this shard's "
                            f"{int(n_local)} valid steps: perm is not a permutation of range({n_total})")
    return ids, offsets


def adam_step(params, grad, exp_avg, exp_avg_sq, step, lr, beta1=0.9, beta2=0.999, eps=1e-8):
    lib = L.load()
    for t, nm in ((params, "params"), (grad, "grad"), (exp_avg, "exp_avg"), (exp_avg_sq, "exp_avg_sq")):
        _need(t, torch.float32, nm, (params.numel(),))
    with torch.cuda.device(params.device):
        rc = lib.tg_adam_step(L.ctx(params.device), params.numel(), L.ptr(params), L.ptr(grad), L.ptr(exp_avg),
                              L.ptr(exp_avg_sq), int(step), float(lr), float(beta1), float(beta2), float(eps),
                              L.stream_ptr())
    L.check(rc, "tg_adam_step")
    _count(1)


def export_trajectory(obs, act, length):
    """tg_export_trajectory: obs [T,O,N], act [T,A,N], len [N] -> (episode_id [n_valid] i32,
    rows [n_valid, O+A] f32) with the valid steps of episode n in rows row0[n] .. row0[n]+len[n]."""
    lib = L.load()
    _need(obs, torch.float32, "obs")
    T, O, N = obs.shape
    A = act.shape[1]
    _need(act, torch.float32, "act", (T, A, N))
    _need(length, torch.int32, "len", (N,))
    dev = obs.device
    csum = torch.cumsum(length.to(torch.int64), 0)
    row0 = (csum - length).contiguous()
    n_valid = int(csum[-1].item())
    ids = torch.empty((n_valid,), dtype=torch.int32, device=dev)
    rows = torch.empty((n_valid, O + A), dtype=torch.float32, device=dev)
    if n_valid > 0:
        with torch.cuda.device(dev):
            rc = lib.tg_export_trajectory(L.ctx(dev), N, T, O, A, L.ptr(obs), L.ptr(act), L.ptr(length), L.ptr(row0),
                                          L.ptr(ids), L.ptr(rows), L.stream_ptr())
        L.check(rc, "tg_export_trajectory")
        _count(1)
    return ids, rows


class _DevMem:
    """A window of C-allocated device memory exposed to torch through __cuda_array_interface__."""

    def __init__(self, ptr: int, n_floats: int):
        self.__cuda_array_interface__ = {"shape": (n_floats,), "typestr": "<f4", "data": (ptr, False), "version": 2}


class PeerComm:
    """tg_comm_*: this rank's gradient window + its peers', for tg_allreduce_adam_step.

    Built collectively by all ranks of an initialised torch.distributed process group (the IPC handles travel through
    all_gather_object).  `grad_slot()` is a torch view of the slot the next step will sum -- pass it as `out_grad` to
    policy_grad / value_grad so the gradient is produced in place."""

    def __init__(self, n_floats: int, device=None):
        import torch.distributed as dist
        lib = L.load()
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.rank, self.world, self.n = dist.get_rank(), dist.get_world_size(), int(n_floats)
        hb = lib.tg_comm_handle_bytes()
        handle = C.create_string_buffer(hb)
        self._h = L._vp()
        err = None
        with torch.cuda.device(self.dev):
            rc = lib.tg_comm_create(L.ctx(self.dev), self.rank, self.world, self.n, C.byref(self._h), handle)
        if rc != 0:
            err = "tg_comm_create: " + lib.tg_last_error().decode(errors="replace")
            self._h = None
        allh = [None] * self.world                       # every rank takes part in both exchanges, failed or not
        dist.all_gather_object(allh, (err, bytes(handle.raw)))
        if all(a[0] is None for a in allh):
            blob = C.create_string_buffer(b"".join(a[1] for a in allh), hb * self.world)
            with torch.cuda.device(self.dev):
                rc = lib.tg_comm_connect(self._h, blob)
            if rc != 0:
                err = "tg_comm_connect: " + lib.tg_last_error().decode(errors="replace")
        else:
            err = err or next(a[0] for a in allh if a[0] is not None)
        errs = [None] * self.world
        dist.all_gather_object(errs, err)
        bad = next((x for x in errs if x is not None), None)
        if bad is not None:
            self.close()
            raise L.EngineError("peer-memory gradient window unavailable: " + bad)

    @staticmethod
    def try_create(n_floats: int, device=None):
        """Collective constructor that cannot leave the ranks disagreeing: every rank reports whether its window
        was created and mapped; unless ALL succeeded, every rank drops its window and None is returned (the caller
        then uses the NCCL allreduce)."""
        import torch.distributed as dist
        comm, err = None, None
        try:
            comm = PeerComm(n_floats, device)
        except Exception as ex:  # noqa: BLE001  (EngineError: no P2P access, IPC refused, ...)
            err = repr(ex)
        oks = [None] * dist.get_world_size()
        dist.all_gather_object(oks, err)
        if any(o is not None for o in oks):
            if comm is not None:
                comm.close()
            PeerComm.last_failure = next(o for o in oks if o is not None)
            return None
        return comm

    last_failure = None

    def grad_slot(self) -> torch.Tensor:
        p = L._vp()
        L.check(L.load().tg_comm_grad_slot(self._h, C.byref(p)), "tg_comm_grad_slot")
        return torch.as_tensor(_DevMem(p.value, self.n), device=self.dev)

    def allreduce_adam_step(self, params, exp_avg, exp_avg_sq, step, lr, beta1=0.9, beta2=0.999, eps=1e-8, out_sum=None):
        lib = L.load()
        n = params.numel()
        for t, nm in ((params, "params"), (exp_avg, "exp_avg"), (exp_avg_sq, "exp_avg_sq")):
            _need(t, torch.float32, nm, (n,))
        with torch.cuda.device(self.dev):
            rc = lib.tg_allreduce_adam_step(L.ctx(self.dev), self._h, n, L.ptr(params), L.ptr(exp_avg), L.ptr(exp_avg_sq),
                                            int(step), float(lr), float(beta1), float(beta2), float(eps), L.ptr(out_sum),
                                            L.stream_ptr())
        L.check(rc, "tg_allreduce_adam_step")
        _count(2)

    def close(self):
        if self._h:
            L.load().tg_comm_destroy(self._h)
            self._h = None
