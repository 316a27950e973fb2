"""tcgen05 building blocks (descriptors, SWIZZLE_128B operand layout, TMEM load) pinned against a
float64 matmul before the fused kernels rely on them."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _run(K, N, passes, seed=0, mode=0):
    from trajopt_grpo_b200 import _lib as L
    lib = L.load()
    rng = np.random.default_rng(seed)
    if mode in (0, 4):  # D[128,N] = A[128,K] @ B[N,K]^T   (mode 4: A operand through tensor memory)
        A = rng.standard_normal((128, K)).astype(np.float32)
        B = rng.standard_normal((N, K)).astype(np.float32)
        ref = A.astype(np.float64) @ B.astype(np.float64).T
    elif mode == 1:    # D[128,N] = A[128,K] @ B[K,N]
        A = rng.standard_normal((128, K)).astype(np.float32)
        B = rng.standard_normal((K, N)).astype(np.float32)
        ref = A.astype(np.float64) @ B.astype(np.float64)
    else:              # D[64,N] = A[K,64]^T @ B[K,N]
        A = rng.standard_normal((K, 64)).astype(np.float32)
        B = rng.standard_normal((K, N)).astype(np.float32)
        ref = A.astype(np.float64).T @ B.astype(np.float64)
    dA, dB = torch.from_numpy(A).cuda(), torch.from_numpy(B).cuda()
    dD = torch.full(ref.shape, float("nan"), device="cuda")
    rc = lib.tg_umma_selftest(L.ctx(), dA.data_ptr(), dB.data_ptr(), dD.data_ptr(), K, N, passes, mode,
                              L.stream_ptr())
    L.check(rc, "tg_umma_selftest")
    torch.cuda.synchronize()
    return dD.cpu().numpy(), ref


@pytest.mark.parametrize("K,N", [(32, 64), (64, 64), (128, 64), (64, 128), (32, 256), (64, 16)])
def test_umma_tf32_single_pass(K, N):
    got, ref = _run(K, N, 1)
    # plain TF32: 10-bit mantissa operands -> ~1e-3 relative to the row scale
    assert np.isfinite(got).all()
    assert np.abs(got - ref).max() <= 4e-3 * np.sqrt(K) * 3


@pytest.mark.parametrize("K,N", [(32, 64), (64, 64), (128, 64), (64, 128), (32, 256), (64, 16)])
def test_umma_3xtf32_is_fp32_faithful(K, N):
    got, ref = _run(K, N, 3, seed=1)
    # 3xTF32 split + truncating fp32 accumulation in the tensor core: ~1e-6 of the row scale per
    # 8 accumulation steps (measured: rms 5.6e-6 at K=64, 1.5e-5 at K=128 for unit-variance data)
    assert np.abs(got - ref).max() <= 1e-6 * K, np.abs(got - ref).max()


@pytest.mark.parametrize("mode,K,N", [(1, 64, 64), (1, 128, 64), (2, 128, 64), (2, 64, 64), (2, 128, 32),
                                      (4, 64, 64), (4, 32, 128)])
def test_umma_mn_major_operands(mode, K, N):
    """backward-data (B MN-major) and weight-gradient (A and B MN-major, M = 64) arrangements"""
    got, ref = _run(K, N, 3, seed=2, mode=mode)
    assert np.isfinite(got).all()
    assert np.abs(got - ref).max() <= 1e-6 * K, np.abs(got - ref).max()


# ----------------------------------------------------------------------------
# fused rollout on the tensor-core path vs the FP32 path and vs the oracle
# ----------------------------------------------------------------------------
def _policy(rng, dims):
    Ws = [(rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(dims[i])).astype(np.float32) for i in range(len(dims) - 1)]
    bs = [(0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32) for i in range(len(dims) - 1)]
    flat = np.concatenate([np.concatenate([w.reshape(-1), b]) for w, b in zip(Ws, bs)]).astype(np.float32)
    return Ws, bs, torch.from_numpy(flat).cuda()


@pytest.mark.parametrize("kind,hidden", [(1, [64, 64]), (3, [64, 64]), (2, [64, 64, 64]), (0, [64, 64]),
                                         (2, [128, 128]), (3, [128, 128]), (1, [128, 128]), (0, [128, 128]),
                                         (3, [256, 256]), (2, [256, 256]), (1, [256, 256]), (0, [256, 256])])
def test_rollout_tensor_core_path_matches_fp32_path_and_oracle(kind, hidden):
    import restate as R
    from trajopt_grpo_b200 import engine as E
    rng = np.random.default_rng(kind)
    O, A = R.OBS_DIM[kind], R.ACT_DIM[kind]
    dims = [O] + hidden + [A]
    Ws, bs, params = _policy(rng, dims)
    N, T = 300, 16
    init = R.reset_states(kind, N, rng)
    noise = rng.standard_normal((T, N, A)).astype(np.float32)
    cov = np.full(A, 0.3, np.float32)
    cfg = R.EnvCfg.make(kind, T)
    o, a, r, lp, ln, m = R.rollout(cfg, init, Ws, bs, cov, noise, dtype=np.float64)
    nz = torch.from_numpy(np.ascontiguousarray(noise.transpose(0, 2, 1))).cuda()
    s0 = torch.from_numpy(init.T.copy()).cuda()
    outs = {}
    try:
        for mode in ("fp32", "3xtf32"):
            E.set_math(mode)
            outs[mode] = E.rollout(kind, T, cfg.dt, dims, "ReLU", params, cov.tolist(), s0, noise=nz)
            torch.cuda.synchronize()
    finally:
        E.set_math("auto")
    for mode, out in outs.items():
        assert np.array_equal(out["len"].cpu().numpy(), ln), mode
        np.testing.assert_allclose(out["obs"].cpu().numpy().transpose(2, 0, 1), o, rtol=1e-4, atol=1e-4, err_msg=mode)
        np.testing.assert_allclose(out["act"].cpu().numpy().transpose(2, 0, 1), a, rtol=1e-4, atol=1e-4, err_msg=mode)
        np.testing.assert_allclose(out["logp"].cpu().numpy().T, lp, rtol=1e-4, atol=1e-4, err_msg=mode)
    # first step (no accumulated drift): the mean action of the two paths agrees to 3xTF32 accuracy
    a32, atc = outs["fp32"]["act"][0].cpu().numpy(), outs["3xtf32"]["act"][0].cpu().numpy()
    assert np.abs(a32 - atc).max() <= 2e-5 * max(1.0, np.abs(a32).max())


@pytest.mark.parametrize("hidden,act_name,N", [([256, 256], "Tanh", 129), ([128, 128], "Sigmoid", 1), ([256, 256], "Sigmoid", 257)])
def test_rollout_wide_tensor_core_kernels_other_activations_and_ragged_tiles(hidden, act_name, N):
    """The 128- and 256-wide tensor-core rollout kernels with non-ReLU activations and env counts that leave
    a partial last tile, against the FP32-pipe kernel (first step: no accumulated drift) and bit-exact
    determinism of repeated launches."""
    import restate as R
    from trajopt_grpo_b200 import engine as E
    kind = 3
    rng = np.random.default_rng(N)
    O, A = R.OBS_DIM[kind], R.ACT_DIM[kind]
    dims = [O] + hidden + [A]
    Ws, bs, params = _policy(rng, dims)
    T = 6
    init = R.reset_states(kind, N, rng)
    noise = rng.standard_normal((T, N, A)).astype(np.float32)
    nz = torch.from_numpy(np.ascontiguousarray(noise.transpose(0, 2, 1))).cuda()
    s0 = torch.from_numpy(init.T.copy()).cuda().float()
    outs = {}
    try:
        for mode in ("fp32", "3xtf32", "3xtf32"):
            E.set_math(mode)
            out = E.rollout(kind, T, 0.02, dims, act_name, params, [0.3] * A, s0, noise=nz)
            torch.cuda.synchronize()
            outs.setdefault(mode, []).append(out)
    finally:
        E.set_math("auto")
    a, b = outs["3xtf32"]
    for k in ("obs", "act", "rew", "logp", "len", "ret"):
        assert torch.equal(a[k], b[k]), k
    f = outs["fp32"][0]
    assert torch.equal(f["len"], a["len"])
    d = (f["act"][0] - a["act"][0]).abs().max().item()
    assert d <= 2e-5 * max(1.0, f["act"][0].abs().max().item()), d
    np.testing.assert_allclose(a["obs"].cpu().numpy(), f["obs"].cpu().numpy(), rtol=2e-3, atol=2e-3)


def test_math_mode_3xtf32_rejects_ineligible_shape():
    from trajopt_grpo_b200 import engine as E
    from trajopt_grpo_b200._lib import EngineError
    params = torch.zeros(3 * 32 + 32 + 32 * 1 + 1, device="cuda")
    try:
        E.set_math("3xtf32")
        with pytest.raises(EngineError, match="not eligible"):
            E.rollout(1, 5, 0.05, [3, 32, 1], "ReLU", params, [0.5], torch.zeros(3, 8, device="cuda"))
    finally:
        E.set_math("auto")


@pytest.mark.parametrize("kind,act_name,width", [(1, "ReLU", 64), (0, "Tanh", 64), (2, "ReLU", 64), (3, "Sigmoid", 64),
                                                 (2, "ReLU", 128), (3, "ReLU", 256), (1, "Tanh", 128), (0, "Sigmoid", 256),
                                                 (3, "Tanh", 128), (2, "Sigmoid", 256)])
def test_policy_grad_tensor_core_path_matches_fp32_path_and_oracle(kind, act_name, width):
    """tg_policy_grad on the tcgen05 paths (O-64-64-A fused kernel; O-128-128-A and O-256-256-A streamed two-kernel
    path) vs the FP32-pipe path and torch float64 autograd,
    ragged episode lengths, two updates' worth of ratio != 1 (old weights differ from current)."""
    import restate as R
    from trajopt_grpo_b200 import engine as E
    rng = np.random.default_rng(10 + kind)
    O, A = R.OBS_DIM[kind], R.ACT_DIM[kind]
    dims = [O, width, width, A]
    Ws, bs, params = _policy(rng, dims)
    oldWs = [w + 0.02 * rng.standard_normal(w.shape).astype(np.float32) for w in Ws]
    G, Eps, T = 5, 52, 9                       # 260 envs: three tiles per step, the last one partial
    N = G * Eps
    obs = rng.standard_normal((G, Eps, T, O)).astype(np.float32)
    actn = rng.standard_normal((G, Eps, T, A)).astype(np.float32)
    adv = rng.standard_normal((G, Eps, T)).astype(np.float32)
    ln = rng.integers(1, T + 1, (G, Eps)).astype(np.int32)
    mask = (np.arange(T)[None, None, :] < ln[:, :, None]).astype(np.float32)
    cov = np.full(A, 0.4, np.float32)
    J, dW, db, lp, old_lp = R.grpo_objective_and_grad(obs, actn, adv * mask, mask, Ws, bs, oldWs, bs, cov, 0.2,
                                                       act=R.ACT_IDS[act_name], dtype="float64")
    ref = np.concatenate([np.concatenate([w.reshape(-1), b]) for w, b in zip(dW, db)])
    dobs = torch.from_numpy(np.ascontiguousarray(obs.reshape(N, T, O).transpose(1, 2, 0))).cuda()
    dact = torch.from_numpy(np.ascontiguousarray(actn.reshape(N, T, A).transpose(1, 2, 0))).cuda()
    dadv = torch.from_numpy(np.ascontiguousarray((adv * mask).reshape(N, T).T)).cuda()
    dlen = torch.from_numpy(ln.reshape(-1)).cuda()
    old_flat = torch.from_numpy(np.concatenate([np.concatenate([w.reshape(-1), b]) for w, b in zip(oldWs, bs)]).astype(np.float32)).cuda()
    out = {}
    try:
        for mode in ("fp32", "3xtf32"):
            E.set_math(mode)
            _, olp = E.policy_forward_traj(dims, act_name, old_flat, dobs, cov.tolist(), dact, dlen)
            g, st = E.policy_grad(dims, act_name, params, cov.tolist(), dobs, dact, dadv, olp, dlen, 0.2, 1.0 / G)
            torch.cuda.synchronize()
            out[mode] = (g.cpu().numpy(), st.cpu().numpy())
    finally:
        E.set_math("auto")
    scale = np.abs(ref).max()
    for mode, (g, st) in out.items():
        assert np.abs(g - ref).max() <= 2e-4 * scale, (mode, np.abs(g - ref).max(), scale)
        assert int(st[1]) == int(mask.sum()), mode
        assert abs(st[0] - J) <= 2e-4 * max(1.0, abs(J)), (mode, st[0], J)
    assert np.abs(out["fp32"][0] - out["3xtf32"][0]).max() <= 5e-5 * scale


@pytest.mark.parametrize("O,width,act_name", [(10, 128, "ReLU"), (20, 256, "ReLU"), (20, 128, "Tanh"),
                                              (3, 128, "ReLU"), (3, 256, "ReLU"), (5, 128, "ReLU"), (5, 256, "ReLU"),
                                              (10, 256, "ReLU"), (20, 128, "ReLU")])
def test_value_grad_wide_tensor_core_path_matches_fp32_path(O, width, act_name):
    """tg_value_grad (critic MSE, ppo.py:168-169) for every built 128/256-wide critic instance on the streamed
    tensor-core path vs the FP32-pipe kernel and torch float64 autograd of c1 * MSE over the valid rows, ragged
    lengths: gradient within GRAD_TOL_F64 of max|g|, sum of squared errors to 1e-5, the valid count exact."""
    import restate as R
    from test_gpu_baseline_shapes import GRAD_TOL_F64, KINK
    from trajopt_grpo_b200 import engine as E
    rng = np.random.default_rng(O + width)
    dims = [O, width, width, 1]
    Ws, bs, _ = _policy(rng, dims)
    N, T = 300, 7
    obs = rng.standard_normal((T, O, N)).astype(np.float32)
    tgt = rng.standard_normal((T, N)).astype(np.float32)
    ln = rng.integers(1, T + 1, N).astype(np.int32)
    mask = (np.arange(T)[:, None] < ln[None, :])
    if act_name == "ReLU":               # no valid sample within fp32 summation noise of a kink
        bs = R.kink_free_biases(obs.transpose(0, 2, 1)[mask], Ws, bs, R.ACT_RELU, KINK)
    params = torch.from_numpy(np.concatenate([np.concatenate([w.reshape(-1), b]) for w, b in zip(Ws, bs)])).cuda()
    scale = 0.5 / mask.sum()
    # float64 reference
    tW = [torch.tensor(w, dtype=torch.float64, requires_grad=True) for w in Ws]
    tb = [torch.tensor(b, dtype=torch.float64, requires_grad=True) for b in bs]
    x = torch.tensor(obs.transpose(0, 2, 1).reshape(T * N, O), dtype=torch.float64)
    actf = {"ReLU": torch.relu, "Tanh": torch.tanh}[act_name]
    h = actf(x @ tW[0].T + tb[0]); h = actf(h @ tW[1].T + tb[1]); v = (h @ tW[2].T + tb[2]).reshape(T, N)
    sq = (((v - torch.tensor(tgt, dtype=torch.float64)) ** 2) * torch.tensor(mask)).sum()
    (scale * sq).backward()
    sse = float(sq.detach())
    ref = np.concatenate([np.concatenate([w.grad.numpy().reshape(-1), b.grad.numpy()]) for w, b in zip(tW, tb)])
    dobs, dtgt, dlen = torch.from_numpy(obs).cuda(), torch.from_numpy(tgt).cuda(), torch.from_numpy(ln).cuda()
    out = {}
    try:
        for mode in ("fp32", "3xtf32"):
            E.set_math(mode)
            g, st = E.value_grad(dims, act_name, params, dobs, dtgt, dlen, scale)
            torch.cuda.synchronize()
            out[mode] = (g.cpu().numpy(), st.cpu().numpy().astype(np.float64))
    finally:
        E.set_math("auto")
    sc = np.abs(ref).max()
    for mode, (g, st) in out.items():
        err = float(np.abs(g - ref).max() / sc)
        e_sse = abs(st[0] - sse) / sse
        print(f"[ppo-parity] value head ({O},1) W {width} {act_name:4s} {mode:6s} grad {err:.2e} "
              f"(<= {GRAD_TOL_F64[mode]:.0e})  sum err^2 {e_sse:.1e} (<= 1e-5)")
        assert err <= GRAD_TOL_F64[mode], (mode, err)
        assert e_sse <= 1e-5, (mode, st[0], sse)
        assert int(st[1]) == int(mask.sum()), mode
    assert np.abs(out["fp32"][0] - out["3xtf32"][0]).max() <= 5e-5 * sc


def test_wide_update_spans_several_scratch_batches():
    """The streamed 128-wide update at a size whose tiles do not fit one scratch batch (6,400 tiles of ~200 KB
    against a 256 MB budget set through TG_TCW_SCRATCH_MB: five batches), ragged lengths: gradient and statistics vs
    the FP32-pipe kernel, and run-to-run determinism."""
    from trajopt_grpo_b200 import engine as E
    rng = np.random.default_rng(77)
    O, A, W = 10, 2, 128
    dims = [O, W, W, A]
    Ws, bs, params = _policy(rng, dims)
    N, T = 4096, 200
    gen = torch.Generator(device="cuda").manual_seed(5)
    obs = torch.randn((T, O, N), device="cuda", generator=gen)
    act = torch.randn((T, A, N), device="cuda", generator=gen)
    adv = torch.randn((T, N), device="cuda", generator=gen)
    olp = -1.5 + 0.1 * torch.randn((T, N), device="cuda", generator=gen)
    ln = torch.randint(1, T + 1, (N,), device="cuda", generator=gen, dtype=torch.int32)
    import os
    os.environ["TG_TCW_SCRATCH_MB"] = "256"
    out = {}
    try:
        for mode in ("fp32", "3xtf32", "3xtf32"):
            E.set_math(mode)
            g, st = E.policy_grad(dims, "ReLU", params, [0.4, 0.4], obs, act, adv, olp, ln, 0.2, 1.0 / 256)
            torch.cuda.synchronize()
            out.setdefault(mode, []).append((g.clone(), st.clone()))
    finally:
        os.environ.pop("TG_TCW_SCRATCH_MB", None)
        E.set_math("auto")
    (g1, s1), (g2, s2) = out["3xtf32"]
    assert torch.equal(g1, g2) and torch.equal(s1, s2)            # deterministic
    gf, sf = out["fp32"][0]
    assert int(s1[1]) == int(ln.sum()) == int(sf[1])
    scale = gf.abs().max().item()
    assert (g1 - gf).abs().max().item() <= 2e-4 * scale
    assert abs(float(s1[0]) - float(sf[0])) <= 2e-4 * max(1.0, abs(float(sf[0])))


def test_tmem_probe_reports_cheap_tensor_memory_accesses():
    """tg_tmem_probe (the microbenchmark behind DESIGN's issue-cost rule): a tcgen05.ld / st pair stays cheap with
    MMAs in flight, and the MMAs retire in a time that grows with their number."""
    import ctypes as C
    from trajopt_grpo_b200 import _lib as L
    lib = L.load()
    res = {}
    for n in (0, 48, -48):
        out = (C.c_longlong * 4)()
        L.check(lib.tg_tmem_probe(L.ctx(torch.device("cuda", 0)), n, out), "tg_tmem_probe")
        res[n] = list(out)
    assert 0 < res[48][0] < 500 and 0 < res[48][1] < 1000          # ld, st(+wait) clocks
    assert res[48][2] > res[0][2]                                    # 48 MMAs take longer than none
    assert res[-48][3] < res[48][3]                                  # warp-uniform issue is cheaper than the lane-0 branch


@pytest.mark.parametrize("O,A,width,act_name", [(10, 2, 128, "ReLU"), (20, 4, 256, "Tanh"), (20, 1, 256, "ReLU")])
def test_policy_forward_traj_wide_tensor_core_path_matches_fp32_path(O, A, width, act_name):
    """tg_policy_forward_traj (critic values / old log-probs over a rollout) for 128/256-wide nets on the streamed
    tensor-core forward vs the FP32-pipe kernel; ragged lengths, rows past the length stay zero."""
    from trajopt_grpo_b200 import engine as E
    rng = np.random.default_rng(O * A + width)
    dims = [O, width, width, A]
    Ws, bs, params = _policy(rng, dims)
    N, T = 333, 6
    obs = torch.from_numpy(rng.standard_normal((T, O, N)).astype(np.float32)).cuda()
    act = torch.from_numpy(rng.standard_normal((T, A, N)).astype(np.float32)).cuda()
    ln = torch.from_numpy(rng.integers(1, T + 1, N).astype(np.int32)).cuda()
    out = {}
    try:
        for mode in ("fp32", "3xtf32"):
            E.set_math(mode)
            mu, lp = E.policy_forward_traj(dims, act_name, params, obs, [0.3] * A, act, ln, want_mu=True, want_logp=True)
            torch.cuda.synchronize()
            out[mode] = (mu.clone(), lp.clone())
    finally:
        E.set_math("auto")
    mask = (torch.arange(T, device="cuda")[:, None] < ln[None, :])
    for k in (0, 1):
        a32, atc = out["fp32"][k], out["3xtf32"][k]
        assert (a32 - atc).abs().max().item() <= 2e-5 * max(1.0, a32.abs().max().item())
    assert float(out["3xtf32"][1][~mask].abs().max()) == 0.0
    assert float(out["3xtf32"][0].permute(0, 2, 1)[~mask].abs().max()) == 0.0
