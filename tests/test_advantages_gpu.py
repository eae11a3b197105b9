"""The advantage kernels (csrc/ssd_advantages.cu) against the float64 oracle (oracle/advantage_ref.py), on the GPU.

Every comparison holds the kernel to oracle.advantage_ref.error_bound: c (T - t + 1) 2^-24 times the recurrence run on
magnitudes (c = 10 + max |log rho|), derived in its docstring and in DESIGN.md section 5.8, not fitted.  With 148 SMs the call
splits time into chunks (C > 1) for M <= 320 at T >= 100 and runs one pass (C = 1) at M = 327 680; both run below."""
import numpy as np
import pytest
import torch

from oracle import advantage_ref as ref

pytestmark = pytest.mark.gpu

GAMMA, LAMBDA, W = 0.97, 0.9, 0.37
MAX_ORACLE_COLUMNS = 400


def _n_for(m):
    return next(n for n in (5, 4, 3, 1) if m % n == 0)


def _dones(pattern, t_count, b, gen):
    d = torch.zeros((t_count, b), dtype=torch.uint8, device="cuda")
    if pattern == "random":
        d = (torch.rand((t_count, b), generator=gen, device="cuda") < 0.03).to(torch.uint8)
    elif pattern == "all_at_one_t":
        d[t_count // 2] = 1
    elif pattern == "t0":
        d[0] = 1
    elif pattern == "last":
        d[t_count - 1] = 1
    elif pattern == "consecutive":
        d[t_count // 3: t_count // 3 + 3] = 1
        d[t_count - 2:] = 1
    else:
        assert pattern == "none"
    return d


def make_inputs(t_count, m, seed=0, reward_dtype=torch.int32, intrinsic=True, pattern="random", n=None):
    n = n or _n_for(m)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    rnd = lambda: torch.randn((t_count, m), generator=gen, device="cuda")
    if reward_dtype == torch.int32:
        rewards = torch.randint(-1, 3, (t_count, m), generator=gen, device="cuda", dtype=torch.int32)
    else:
        rewards = rnd()
    return dict(rewards=rewards, values=rnd(), dones=_dones(pattern, t_count, m // n, gen),
                bootstrap=torch.randn((m,), generator=gen, device="cuda"),
                intrinsic=torch.rand((t_count, m), generator=gen, device="cuda") if intrinsic else None,
                target_logp=0.6 * rnd() - 1.5, behaviour_logp=0.6 * rnd() - 1.5)


def _columns(m):
    if m <= MAX_ORACLE_COLUMNS:
        return np.arange(m)
    rng = np.random.RandomState(m)
    return np.unique(np.concatenate([np.arange(8), rng.choice(m, 240, replace=False), np.arange(m - 16, m)]))


def _host(x, cols, n=None):
    """Columns `cols` of a [T, M] tensor (or [M]) as numpy; dones [T, B] become the [T, len(cols)] dones of those columns."""
    if x is None:
        return None
    idx = torch.as_tensor(cols if n is None else cols // n, device=x.device)
    return x.index_select(x.dim() - 1, idx).cpu().numpy()


def run(mode, inp, **kw):
    from sequential_social_dilemma_games_b200 import postprocess
    common = dict(intrinsic=inp["intrinsic"], intrinsic_weight=W)
    common.update({k: v for k, v in kw.items() if k in ("intrinsic", "intrinsic_weight")})
    args = (inp["rewards"], inp["values"], inp["dones"], inp["bootstrap"])
    if mode == "gae":
        return postprocess.compute_advantages(*args, gamma=kw.get("gamma", GAMMA), lambda_=kw.get("lambda_", LAMBDA), **common)
    if mode == "returns":
        return postprocess.compute_advantages(*args, gamma=kw.get("gamma", GAMMA), lambda_=LAMBDA, use_gae=False, **common)
    return tuple(postprocess.vtrace(*args, inp["target_logp"], inp["behaviour_logp"], gamma=kw.get("gamma", GAMMA),
                                    clip_rho_threshold=kw.get("rho", 1.0), clip_pg_rho_threshold=kw.get("pg", float("inf")), **common))


def check(mode, inp, out, **kw):
    """Compares the kernel's outputs on sampled columns with the oracle; returns the largest error relative to its bound."""
    m = inp["values"].shape[1]
    n = m // inp["dones"].shape[1]
    cols = _columns(m)
    h = {k: _host(v, cols) for k, v in inp.items() if k != "dones"}
    d = _host(inp["dones"], cols, n)
    intr, w = (h["intrinsic"], W) if inp["intrinsic"] is not None else (None, 0.0)
    gamma, lam, rho, pg = kw.get("gamma", GAMMA), kw.get("lambda_", LAMBDA), kw.get("rho", 1.0), kw.get("pg", np.inf)
    if mode == "vtrace":
        want = ref.vtrace(h["rewards"], h["values"], d, h["bootstrap"], h["target_logp"], h["behaviour_logp"], gamma, rho, pg, intr, w)
        bound = ref.error_bound("vtrace", h["rewards"], h["values"], d, h["bootstrap"], gamma, 1.0, intr, w, h["target_logp"],
                                h["behaviour_logp"], rho, pg)
    else:
        want = ref.compute_advantages(h["rewards"], h["values"], d, h["bootstrap"], gamma, lam, mode == "gae", intr, w)
        bound = ref.error_bound(mode, h["rewards"], h["values"], d, h["bootstrap"], gamma, lam, intr, w)
    worst = 0.0
    for name, got, exp, tol in zip(("out0", "out1"), out, want, bound):
        if exp is None:
            assert got is None
            continue
        g = got.reshape(got.shape[0], -1)[:, torch.as_tensor(cols, device=got.device)].double().cpu().numpy()
        err = np.abs(g - exp)
        assert np.isfinite(g).all(), (mode, name)
        bad = err > tol
        assert not bad.any(), "%s %s: %d elements above the bound, worst err %.3g at bound %.3g" % (
            mode, name, bad.sum(), err[bad].max(), tol[bad][err[bad].argmax()])
        worst = max(worst, float((err / np.maximum(tol, 1e-300)).max()))
    return worst


SHAPES = [(t, m) for t in (1, 2, 7, 100, 1000) for m in (1, 5, 127, 128, 129, 320, 327680)]


@pytest.mark.parametrize("t_count,m", SHAPES, ids=["T%d-M%d" % s for s in SHAPES])
def test_shapes_against_oracle(t_count, m):
    k = SHAPES.index((t_count, m))
    patterns = ("random", "none", "all_at_one_t", "t0", "last", "consecutive")
    inp = make_inputs(t_count, m, seed=k, reward_dtype=(torch.int32, torch.float32)[k % 2], intrinsic=k % 3 != 0,
                      pattern=patterns[k % len(patterns)])
    worst = {mode: check(mode, inp, run(mode, inp)) for mode in ("gae", "returns", "vtrace")}
    print("T=%d M=%d max err / bound %s" % (t_count, m, {k: "%.3g" % v for k, v in worst.items()}))


PATHS = [(1000, 320), (100, 327680)]   # C > 1 and C = 1


@pytest.mark.parametrize("t_count,m", PATHS, ids=["chunked", "single"])
@pytest.mark.parametrize("reward_dtype", [torch.int32, torch.float32], ids=["i32", "f32"])
@pytest.mark.parametrize("intrinsic", [True, False], ids=["intrinsic", "extrinsic"])
@pytest.mark.parametrize("mode", ["gae", "returns", "vtrace"])
def test_modes_dtypes_intrinsic(mode, intrinsic, reward_dtype, t_count, m):
    inp = make_inputs(t_count, m, seed=7, reward_dtype=reward_dtype, intrinsic=intrinsic)
    check(mode, inp, run(mode, inp))


@pytest.mark.parametrize("t_count,m", PATHS, ids=["chunked", "single"])
@pytest.mark.parametrize("pattern", ["none", "all_at_one_t", "random", "t0", "last", "consecutive"])
def test_done_patterns(pattern, t_count, m):
    inp = make_inputs(t_count, m, seed=11, pattern=pattern)
    for mode in ("gae", "returns", "vtrace"):
        check(mode, inp, run(mode, inp))


@pytest.mark.parametrize("t_count,m", PATHS, ids=["chunked", "single"])
@pytest.mark.parametrize("pg", [1.0, 2.0, float("inf")])
@pytest.mark.parametrize("rho", [1.0, 2.0, float("inf")])
def test_clip_thresholds(rho, pg, t_count, m):
    inp = make_inputs(t_count, m, seed=13)
    check("vtrace", inp, run("vtrace", inp, rho=rho, pg=pg), rho=rho, pg=pg)


def test_chunked_columns_equal_the_same_columns_in_one_pass():
    """Envs 0..63 of a 65 536-env call (C = 1) against the same 64 envs alone (C > 1)."""
    big = make_inputs(1000, 327680, seed=17)
    small = {k: (None if v is None else v[..., :320].contiguous() if k != "dones" else v[:, :64].contiguous()) for k, v in big.items()}
    cols = np.arange(320)
    for mode in ("gae", "returns", "vtrace"):
        a, b = run(mode, small), run(mode, big)
        bound = _bounds(mode, small, cols)
        for x, y, tol in zip(a, b, bound):
            if x is None:
                continue
            err = (x - y[:, :320]).abs().double().cpu().numpy()
            assert (err <= 2 * tol).all(), (mode, float(err.max()))


def _bounds(mode, inp, cols, **kw):
    h = {k: _host(v, cols) for k, v in inp.items() if k != "dones"}
    d = _host(inp["dones"], cols, inp["values"].shape[1] // inp["dones"].shape[1])
    intr = h["intrinsic"]
    if mode == "vtrace":
        return ref.error_bound("vtrace", h["rewards"], h["values"], d, h["bootstrap"], kw.get("gamma", GAMMA), 1.0, intr, W,
                               h["target_logp"], h["behaviour_logp"], kw.get("rho", 1.0), kw.get("pg", np.inf))
    return ref.error_bound(mode, h["rewards"], h["values"], d, h["bootstrap"], kw.get("gamma", GAMMA),
                           kw.get("lambda_", LAMBDA), intr, W)


@pytest.mark.parametrize("t_count,m", PATHS, ids=["chunked", "single"])
def test_on_policy_vtrace_is_gae_lambda_one_is_returns(t_count, m):
    inp = make_inputs(t_count, m, seed=19)
    inp["target_logp"] = inp["behaviour_logp"].clone()                 # log rho = 0
    adv1, vt1 = run("gae", inp, lambda_=1.0)
    ret, _ = run("returns", inp)
    vs, pg = run("vtrace", inp, rho=1.0, pg=2.0)
    cols = _columns(m)
    b_gae = _bounds("gae", inp, cols, lambda_=1.0)
    b_ret = _bounds("returns", inp, cols)
    b_vt = _bounds("vtrace", inp, cols, rho=1.0, pg=2.0)
    sel = lambda x: x[:, torch.as_tensor(cols, device=x.device)].double().cpu().numpy()
    assert (np.abs(sel(vs) - sel(vt1)) <= b_vt[0] + b_gae[1]).all()
    assert (np.abs(sel(vt1) - sel(ret)) <= b_gae[1] + b_ret[0]).all()
    assert (np.abs(sel(pg) - sel(adv1)) <= b_vt[1] + b_gae[0]).all()


@pytest.mark.parametrize("t_count,m", PATHS, ids=["chunked", "single"])
def test_repeated_calls_are_bitwise_identical(t_count, m):
    inp = make_inputs(t_count, m, seed=23)
    for mode in ("gae", "returns", "vtrace"):
        a, b = run(mode, inp), run(mode, inp)
        for x, y in zip(a, b):
            assert x is None and y is None or torch.equal(x, y), mode


@pytest.mark.parametrize("t_count,m", PATHS, ids=["chunked", "single"])
def test_non_finite_after_a_done_does_not_reach_earlier_steps(t_count, m):
    inp = make_inputs(t_count, m, seed=29, pattern="random")
    n = m // inp["dones"].shape[1]
    d = inp["dones"].bool()
    has = d.any(0)
    first = torch.where(has, d.float().argmax(0), torch.full_like(has, t_count, dtype=torch.long))   # first done of each env
    t = torch.arange(t_count, device="cuda")[:, None]
    after = (t > first.repeat_interleave(n)[None, :])                                                  # [T, M]: behind that done
    assert after.any() and (~after).any()
    base = {mode: run(mode, inp) for mode in ("gae", "returns", "vtrace")}
    for poison in (float("nan"), float("inf"), -float("inf")):
        bad = dict(inp)
        for k in ("values", "intrinsic", "target_logp", "behaviour_logp"):
            bad[k] = torch.where(after, torch.full_like(inp[k], poison), inp[k])
        bad["rewards"] = inp["rewards"].float().masked_fill(after, poison)      # float(int32 reward) is exact: same r_t before
        ended = has.repeat_interleave(n)
        bad["bootstrap"] = torch.where(ended, torch.full_like(inp["bootstrap"], poison), inp["bootstrap"])
        for mode, ref_out in base.items():
            out = run(mode, bad)
            for x, y in zip(out, ref_out):
                if x is None:
                    continue
                keep = ~after
                assert torch.equal(x[keep], y[keep]), (mode, poison)
                assert torch.isfinite(x[keep]).all()
    # a done at T-1: the bootstrap is never read
    inp = make_inputs(t_count, m, seed=31, pattern="last")
    for mode in ("gae", "returns", "vtrace"):
        a = run(mode, inp)
        for poison in (float("nan"), float("inf")):
            b = run(mode, dict(inp, bootstrap=torch.full_like(inp["bootstrap"], poison)))
            for x, y in zip(a, b):
                assert x is None or torch.equal(x, y), (mode, poison)


def test_index_width_above_2_pow_31():
    """Returns mode with T * M = 2^31 + 32: the last 32 columns of step T-1 sit above element 2^31."""
    t_count, m = 4, 536870920
    need = t_count * m * 4 * 3 + (1 << 30)
    if torch.cuda.mem_get_info()[0] < need:
        pytest.skip("needs %.1f GB of free device memory" % (need / 1e9))
    assert t_count * m > 2 ** 31
    gen = torch.Generator(device="cuda").manual_seed(37)
    inp = dict(rewards=torch.randint(-1, 3, (t_count, m), generator=gen, device="cuda", dtype=torch.int32),
               values=torch.empty((t_count, m), device="cuda"),
               dones=(torch.rand((t_count, m // 5), generator=gen, device="cuda") < 0.2).to(torch.uint8),
               bootstrap=torch.randn((m,), generator=gen, device="cuda"), intrinsic=None)
    adv, vt = run("returns", inp)
    assert vt is None
    cols = np.unique(np.concatenate([np.arange(64), np.random.RandomState(0).choice(m, 512, replace=False), np.arange(m - 64, m)]))
    h_r = inp["rewards"][:, torch.as_tensor(cols, device="cuda")].cpu().numpy()
    h_b = inp["bootstrap"][torch.as_tensor(cols, device="cuda")].cpu().numpy()
    h_d = inp["dones"][:, torch.as_tensor(cols // 5, device="cuda")].cpu().numpy()
    zeros = np.zeros_like(h_r, np.float32)
    want, _ = ref.compute_advantages(h_r, zeros, h_d, h_b, GAMMA, LAMBDA, False)
    tol, _ = ref.error_bound("returns", h_r, zeros, h_d, h_b, GAMMA)
    got = adv[:, torch.as_tensor(cols, device="cuda")].double().cpu().numpy()
    assert (np.abs(got - want) <= tol).all()
    del inp, adv
    torch.cuda.empty_cache()


def test_closed_loop_env_policy_advantages():
    """Harvest, 64 envs x 5 agents, T = 150: env -> policy_step -> env, episodes cut at t = 59 and 119 (env.reset), the value of
    the last observation as bootstrap; then compute_advantages and vtrace against the oracle on the recorded buffers."""
    from sequential_social_dilemma_games_b200 import policy, postprocess
    from sequential_social_dilemma_games_b200.batched import BatchedSSDEnv, make_config
    cfg = make_config("harvest")
    b, n, t_count = 64, cfg.num_agents, 150
    env = BatchedSSDEnv(cfg, b, device="cuda:0", seed=5)
    net = policy.ConvToFCNet(policy.random_weights(num_outputs=cfg.num_actions, seed=1), device="cuda:0")
    target = policy.ConvToFCNet(policy.random_weights(num_outputs=cfg.num_actions, seed=2), device="cuda:0")
    net.seed_sampling(3)
    rewards = torch.empty((t_count, b, n), dtype=torch.int32, device="cuda")
    values = torch.empty((t_count, b, n), device="cuda")
    logp = torch.empty_like(values)
    tlogp = torch.empty_like(values)
    dones = torch.zeros((t_count, b), dtype=torch.uint8, device="cuda")
    obs = env.reset()
    h, c = net.initial_state(b * n)
    ht, ct = target.initial_state(b * n)
    for t in range(t_count):
        s = net.policy_step(obs, h, c)
        st = target.policy_step(obs, ht, ct, mode="given", actions=s.actions)
        values[t], logp[t], tlogp[t] = s.value.view(b, n), s.logp.view(b, n), st.logp.view(b, n)
        obs, _ = env.step(s.actions.view(b, n), reward_out=rewards[t])
        h, c, ht, ct = s.h, s.c, st.h, st.c
        if t in (59, 119):
            dones[t] = 1
            obs = env.reset()
            h, c = net.initial_state(b * n)
            ht, ct = target.initial_state(b * n)
    boot = net.policy_step(obs, h, c, mode="greedy").value.view(b, n)
    adv, vt = postprocess.compute_advantages(rewards, values, dones, boot, gamma=0.99, lambda_=0.95)
    vs, pg = postprocess.vtrace(rewards, values, dones, boot, tlogp, logp, gamma=0.99, clip_rho_threshold=1.0,
                                clip_pg_rho_threshold=1.0)
    assert adv.shape == (t_count, b, n) and vs.shape == (t_count, b, n)
    h = lambda x: x.reshape(t_count, -1).cpu().numpy()
    r_h, v_h, d_h, b_h = h(rewards), h(values), dones.cpu().numpy(), boot.reshape(-1).cpu().numpy()
    assert r_h.any(), "no reward in the closed loop"
    want = ref.compute_advantages(r_h, v_h, d_h, b_h, 0.99, 0.95)
    tol = ref.error_bound("gae", r_h, v_h, d_h, b_h, 0.99, 0.95)
    for got, w_, t_ in zip((adv, vt), want, tol):
        assert (np.abs(h(got) - w_) <= t_).all()
    want = ref.vtrace(r_h, v_h, d_h, b_h, h(tlogp), h(logp), 0.99, 1.0, 1.0)
    tol = ref.error_bound("vtrace", r_h, v_h, d_h, b_h, 0.99, 1.0, None, 0.0, h(tlogp), h(logp), 1.0, 1.0)
    for got, w_, t_ in zip((vs, pg), want, tol):
        assert (np.abs(h(got) - w_) <= t_).all()
    net.close()
    target.close()


def test_python_argument_errors():
    from sequential_social_dilemma_games_b200 import postprocess
    inp = make_inputs(10, 20, seed=41)
    args = (inp["rewards"], inp["values"], inp["dones"], inp["bootstrap"])
    with pytest.raises(TypeError):
        postprocess.compute_advantages(inp["rewards"].double(), *args[1:], gamma=0.9, lambda_=0.9)
    with pytest.raises(ValueError):
        postprocess.compute_advantages(inp["rewards"], inp["values"].t(), *args[2:], gamma=0.9, lambda_=0.9)
    with pytest.raises(ValueError):                                          # the right shape, not contiguous
        postprocess.compute_advantages(inp["rewards"], inp["values"].t().contiguous().t(), *args[2:], gamma=0.9, lambda_=0.9)
    with pytest.raises(ValueError):
        postprocess.compute_advantages(inp["rewards"].cpu(), *args[1:], gamma=0.9, lambda_=0.9)
    with pytest.raises(ValueError):
        postprocess.compute_advantages(*args[:3], inp["bootstrap"][:5], gamma=0.9, lambda_=0.9)
    with pytest.raises(TypeError):
        postprocess.compute_advantages(*args, gamma=0.9)                       # no default for lambda_
    from sequential_social_dilemma_games_b200 import _lib
    with pytest.raises(_lib.SsdError):
        postprocess.compute_advantages(*args, gamma=1.5, lambda_=0.9)
    with pytest.raises(_lib.SsdError):
        postprocess.vtrace(*args, inp["target_logp"], inp["behaviour_logp"], gamma=0.9, clip_rho_threshold=-1.0,
                           clip_pg_rho_threshold=1.0)
    # [T, B, N] and [T, M] give the same result, shaped like values
    a3, v3 = postprocess.compute_advantages(inp["rewards"].view(10, 4, 5), inp["values"].view(10, 4, 5), inp["dones"],
                                            inp["bootstrap"].view(4, 5), gamma=0.9, lambda_=0.8)
    a2, v2 = postprocess.compute_advantages(*args, gamma=0.9, lambda_=0.8)
    assert a3.shape == (10, 4, 5) and torch.equal(a3.view(10, 20), a2) and torch.equal(v3.view(10, 20), v2)
