"""MOA pool (MOAPool, ssd_moa_create_pool / ssd_moa_pool_step): K MOA weight sets, agent m evaluated with set policy_ids[m] of
each call.  Each agent runs the instruction sequence of the shared MOA kernel on its set's weights, so the reference -- K shared
MOANets, each run on ALL M agents, keeping the rows whose id is k -- is matched bitwise; the float64 oracle (oracle/moa_ref.py)
bounds the outputs to the tolerances of test_moa_gpu.py.  Every comparison runs three recurrent steps with the state carried.
Also: policy_step(features=...) of the networks and the policy pool, bitwise equal to the call that runs the trunk."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from test_moa_gpu import MOA_TOL, _inputs, _np, _sets, _weights
from test_policy_pool_gpu import _ids_with_sizes

pytestmark = pytest.mark.gpu

SCALE_B = 65536   # Harvest envs x 5 agents = 327 680 agents per call


def _policy():
    from sequential_social_dilemma_games_b200 import policy
    return policy


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _random_state(m, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return 0.5 * torch.randn((m, 128), device="cuda", generator=g), 0.5 * torch.randn((m, 128), device="cuda", generator=g)


def _rows(pool, s, m):
    """The outputs of an MOAStep as agent-major rows: pred, influence, influence_per_agent, h', c'."""
    return [s.pred, s.influence, s.influence_per_agent, pool.state_rows(s.h, m), pool.state_rows(s.c, m)]


NAMES = ("pred", "influence", "influence_per_agent", "h", "c", "counterfactual")


class RowwiseReference(object):
    """K shared MOANets, each evaluated on all M agents; agent m keeps the outputs of MOA ids[m].  (h, c) are carried as
    agent-major rows."""

    def __init__(self, sets, n):
        self.nets = [_policy().MOANet(w, n) for w in sets]

    def step(self, x, ids, joint, pl, h_rows, c_rows, counterfactuals=False, **kw):
        m = x.shape[0]
        ids = ids.reshape(-1).long()
        out = None
        for k, net in enumerate(self.nets):
            sel = ids == k
            if not bool(sel.any()):
                continue
            s = net.step(x, joint, pl, net.state_from_rows(h_rows), net.state_from_rows(c_rows), counterfactuals=counterfactuals, **kw)
            r = _rows(net, s, m) + ([s.counterfactual] if counterfactuals else [])
            if out is None:
                out = [torch.zeros_like(t) for t in r]
            for o, t in zip(out, r):
                o[sel] = t[sel]
        return out

    def close(self):
        for n in self.nets:
            n.close()


def _check_against_reference(sets, n, steps, ids_per_step, state_seed=1, counterfactuals=False, **kw):
    """Pool vs the row-wise reference over the recurrent steps, bitwise on the agents with an MOA; the reference's state is the
    pool's previous output (so both see the same state at every step).  Returns the pool's steps."""
    policy = _policy()
    m = steps[0][0].shape[0]
    pool = policy.MOAPool(sets, n)
    ref = RowwiseReference(sets, n)
    hr, cr = _random_state(m, state_seed)
    h, c = pool.state_from_rows(hr), pool.state_from_rows(cr)
    got = []
    for t, ((x, joint, pl), ids) in enumerate(zip(steps, ids_per_step)):
        s = pool.step(x, ids, joint, pl, h, c, counterfactuals=counterfactuals, **kw)
        want = ref.step(x, ids, joint, pl, pool.state_rows(h, m), pool.state_rows(c, m), counterfactuals=counterfactuals, **kw)
        live = ids.reshape(-1).long() < len(sets)
        for name, g, w in zip(NAMES, _rows(pool, s, m) + ([s.counterfactual] if counterfactuals else []), want):
            assert torch.equal(g[live], w[live]), (t, name)
        got.append(s)
        h, c = s.h, s.c
    pool.close()
    ref.close()
    return got


@pytest.mark.parametrize("n,a,B", [(5, 8, 1), (5, 8, 25), (5, 9, 26), (5, 8, 27), (5, 8, 1025), (2, 8, 300), (9, 8, 77)])
def test_pool_of_one_equals_shared_moa(n, a, B):
    """M = 5, 125, 130, 135, 5 125: one partial tile, a full tile and a short one, many tiles per call."""
    policy = _policy()
    m = B * n
    w = _weights(n, a, seed=100 + B)
    shared, pool = policy.MOANet(w, n), policy.MOAPool([w], n)
    assert pool.num_policies == 1
    ids = torch.zeros((B, n), dtype=torch.uint8, device="cuda")
    hr, cr = _random_state(m, B)
    hs, cs = shared.state_from_rows(hr), shared.state_from_rows(cr)
    hp, cp = pool.state_from_rows(hr), pool.state_from_rows(cr)
    assert hp.shape == hs.shape and hp.shape == pool.initial_state(m)[0].shape
    cf = B == 1025
    for x, joint, pl in _inputs(B, n, a, seed=B + n):
        s1 = shared.step(x, joint, pl, hs, cs, counterfactuals=cf)
        s2 = pool.step(x, ids, joint, pl, hp, cp, counterfactuals=cf)
        for name, g, want in zip(NAMES, _rows(pool, s2, m), _rows(shared, s1, m)):
            assert torch.equal(g, want), name
        assert (s2.counterfactual is None) == (not cf)
        if cf:
            assert torch.equal(s2.counterfactual, s1.counterfactual)
        hs, cs, hp, cp = s1.h, s1.c, s2.h, s2.c
    shared.close()
    pool.close()


@pytest.mark.parametrize("n", [2, 5, 9])
def test_identity_mapping_equals_per_agent_moa(n):
    policy = _policy()
    a, B = 8, 300
    m = B * n
    sets = _sets(n, a, n, seed=200 + n)
    per, pool = policy.MOANet(sets, n), policy.MOAPool(sets, n)
    ids = torch.arange(n, dtype=torch.uint8, device="cuda").repeat(B, 1)
    hr, cr = _random_state(m, n)
    hq, cq = per.state_from_rows(hr), per.state_from_rows(cr)
    hp, cp = pool.state_from_rows(hr), pool.state_from_rows(cr)
    for x, joint, pl in _inputs(B, n, a, seed=n):
        s1, s2 = per.step(x, joint, pl, hq, cq), pool.step(x, ids, joint, pl, hp, cp)
        for name, g, want in zip(NAMES, _rows(pool, s2, m), _rows(per, s1, m)):
            assert torch.equal(g, want), name
        hq, cq, hp, cp = s1.h, s1.c, s2.h, s2.c
    per.close()
    pool.close()


@pytest.mark.parametrize("K,sizes,a", [
    pytest.param(3, {0: 129, 1: 0}, 8, id="3-sizes0"),                               # policy 2 takes the rest
    pytest.param(3, {1: 1, 2: 127}, 9, id="3-sizes1-cleanup"),
    pytest.param(40, {0: 0, 1: 1, 2: 127, 3: 128, 4: 129}, 8, id="40-sizes2"),
    pytest.param(255, {7: 127, 8: 128, 9: 129, 10: 1, 11: 0}, 8, id="255-sizes3"),
])
def test_random_ids_match_rowwise_reference(K, sizes, a):
    n, B = 5, 1025
    m = B * n
    ids = _ids_with_sizes(m, K, sizes, seed=K + a)
    counts = torch.bincount(ids.long(), minlength=256).cpu().numpy()
    for k, c in sizes.items():
        assert counts[k] == c
    _check_against_reference(_sets(n, a, K, seed=K), n, _inputs(B, n, a, seed=K), [ids] * 3, counterfactuals=K == 40)


def test_one_policy_holds_every_agent():
    n, a, B = 5, 8, 1025
    ids = torch.full((B, n), 17, dtype=torch.uint8, device="cuda")
    _check_against_reference(_sets(n, a, 40, seed=3), n, _inputs(B, n, a, seed=4), [ids] * 3)


def test_scale_many_tiles_per_cta():
    """65 536 Harvest envs x 5 agents, K = 40 random ids: every CTA runs many tiles and reloads weights across policy boundaries."""
    n, a, K = 5, 8, 40
    m = SCALE_B * n
    g = torch.Generator(device="cuda").manual_seed(7)
    ids = torch.randint(0, K, (SCALE_B, n), dtype=torch.uint8, device="cuda", generator=g)
    counts = torch.bincount(ids.reshape(-1).long(), minlength=K).cpu().numpy()
    tiles = sum((int(c) + 127) // 128 for c in counts)
    assert tiles >= 4 * _sms() and tiles > K
    _check_against_reference(_sets(n, a, K, seed=60), n, _inputs(SCALE_B, n, a, seed=8), [ids] * 3)
    assert m == 327680


def test_reassignment_between_steps():
    """New ids at every step on a live state, which stays agent-major."""
    n, a, B, K = 5, 8, 800, 7
    g = torch.Generator(device="cuda").manual_seed(1)
    ids = [torch.randint(0, K, (B, n), dtype=torch.uint8, device="cuda", generator=g) for _ in range(3)]
    assert not torch.equal(ids[0], ids[1])
    _check_against_reference(_sets(n, a, K, seed=70), n, _inputs(B, n, a, seed=2), ids)


def test_skipped_agents_are_not_written():
    policy = _policy()
    from sequential_social_dilemma_games_b200 import _lib
    L = _lib.lib
    n, a, B, K = 5, 8, 400, 4
    m = B * n
    sets = _sets(n, a, K, seed=80)
    pool = policy.MOAPool(sets, n)
    g = torch.Generator(device="cuda").manual_seed(3)
    ids = torch.randint(0, K + 3, (B, n), dtype=torch.uint8, device="cuda", generator=g)
    ids[::37, 2] = 255
    skip = ids.reshape(-1).long() >= K
    assert 0 < int(skip.sum()) < m
    x, joint, pl = _inputs(B, n, a, seed=81, steps=1)[0]
    pl[skip] = float("nan")   # a skipped agent's policy logits are not read
    hr, cr = _random_state(m, 82)
    h, c = pool.state_from_rows(hr), pool.state_from_rows(cr)
    # C level: sentinel-filled outputs keep the sentinel in the skipped rows
    p = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    pred, cf = torch.full((m, n - 1, a), 7.5, device="cuda"), torch.full((m, a, n - 1, a), -7.5, device="cuda")
    ipa, infl = torch.full((m, n - 1), 9.5, device="cuda"), torch.full((m,), -9.5, device="cuda")
    hn, cn = torch.full_like(h, 3.25), torch.full_like(c, -3.25)
    assert L.ssd_moa_pool_step(pool._h, p(x), p(ids), p(joint), p(pl), p(h), p(c), p(hn), p(cn), p(pred), p(cf), p(ipa), p(infl), m, 0,
                               math.inf, st) == 0
    torch.cuda.synchronize()
    assert bool((pred[skip] == 7.5).all()) and bool((cf[skip] == -7.5).all())
    assert bool((ipa[skip] == 9.5).all()) and bool((infl[skip] == -9.5).all())
    assert bool((pool.state_rows(hn, m)[skip] == 3.25).all()) and bool((pool.state_rows(cn, m)[skip] == -3.25).all())
    # the live agents equal the reference, which sees the skipped agents' (scripted) actions among the others
    live = ~skip
    ref = RowwiseReference(sets, n)
    want = ref.step(x, ids, joint, pl, hr, cr, counterfactuals=True)
    for name, got, w in zip(NAMES, [pred, infl, ipa, pool.state_rows(hn, m), pool.state_rows(cn, m), cf], want):
        assert torch.equal(got[live], w[live]), name
    assert bool(torch.isfinite(infl[live]).all())
    # a skipped agent with action -1 makes its env's influence NaN
    mixed = skip.reshape(B, n).any(dim=1) & (~skip).reshape(B, n).any(dim=1)   # envs with a skipped and a live agent
    bad_env = int(torch.nonzero(mixed)[0])
    bad_agent = int(torch.nonzero(skip.reshape(B, n)[bad_env])[0])
    joint2 = joint.clone()
    joint2[bad_env, bad_agent] = -1
    s = pool.step(x, ids, joint2, pl, h, c)
    env_of = torch.arange(m, device="cuda") // n
    in_bad = live & (env_of == bad_env)
    assert bool(in_bad.any()) and bool(torch.isnan(s.influence[in_bad]).all()) and bool(torch.isnan(s.influence_per_agent[in_bad]).all())
    others = live & (env_of != bad_env)
    assert torch.equal(s.influence[others], infl[others])
    want2 = ref.step(x, ids, joint2, pl, hr, cr)
    assert torch.equal(s.pred[live], want2[0][live])   # the others' MOA inputs carry a zero one-hot row for it
    ref.close()
    pool.close()


@pytest.mark.parametrize("divergence,clip", [("kl", math.inf), ("jsd", math.inf), ("kl", 0.02)])
@pytest.mark.parametrize("n,a", [pytest.param(5, 8, id="8"), pytest.param(5, 9, id="9"),
                                 (2, 1), (16, 4), (2, 9), (5, 15)])   # A = 1, N >= 10, (N - 1) A % 4 != 0, A >= 10
def test_matches_float64_oracle(n, a, divergence, clip):
    from oracle import moa_ref
    policy = _policy()
    B, K = 157, 3
    m = B * n
    sets = _sets(n, a, K, seed=90 + a)
    pool = policy.MOAPool(sets, n)
    ids = torch.randint(0, K, (B, n), dtype=torch.uint8, device="cuda", generator=torch.Generator(device="cuda").manual_seed(a))
    idn = ids.reshape(-1).cpu().numpy()
    hr, cr = _random_state(m, 91)
    h, c = pool.state_from_rows(hr), pool.state_from_rows(cr)
    h64, c64 = _np(pool.state_rows(h, m)), _np(pool.state_rows(c, m))
    tol_infl = 8 * MOA_TOL * (n - 1)
    for t, (x, joint, pl) in enumerate(_inputs(B, n, a, seed=92)):
        s = pool.step(x, ids, joint, pl, h, c, divergence=divergence, clip=clip, counterfactuals=True)
        outs = [moa_ref.moa_forward(w, _np(x), _np(joint).astype(np.int64), _np(pl), h64, c64, a, divergence=divergence, clip=clip)
                for w in sets]
        ref = {k: np.stack([outs[idn[r]][k][r] for r in range(m)]) for k in outs[0]}
        for name, got, tol in (("pred", s.pred, MOA_TOL), ("h", pool.state_rows(s.h, m), MOA_TOL), ("c", pool.state_rows(s.c, m), MOA_TOL),
                               ("counterfactual", s.counterfactual, MOA_TOL), ("influence_per_agent", s.influence_per_agent, tol_infl),
                               ("influence", s.influence, tol_infl)):
            err = np.abs(_np(got) - ref[name]).max()
            assert err < tol, (t, name, err)
        if a == 1:   # one action: the influence is exactly 0
            assert bool((s.influence == 0).all())
        else:
            assert np.abs(ref["influence"]).max() > 1e-3   # not vacuous
        if clip < math.inf:
            assert float(s.influence.max()) <= clip
        h, c, h64, c64 = s.h, s.c, ref["h"], ref["c"]
    pool.close()


def test_closed_loop_runs_by_block_mapping():
    """BatchedSSDEnv (300 Harvest envs x 5 agents) -> PolicyPool.features -> PolicyPool.policy_step(features=x) -> MOAPool.step ->
    env.step for six steps; three runs x five agents, env b belongs to run b mod 3: ids[b, n] = 5 (b mod 3) + n for both pools.
    On the recorded observations, actions and logits the MOA outputs equal the row-wise reference's."""
    policy = _policy()
    from sequential_social_dilemma_games_b200.batched import BatchedSSDEnv, make_config
    R, N, B, A = 3, 5, 300, 8
    m = B * N
    ids = (N * (torch.arange(B, device="cuda")[:, None] % R) + torch.arange(N, device="cuda")[None, :]).to(torch.uint8)
    env = BatchedSSDEnv(make_config("harvest", num_agents=N), B, seed=5)
    pool = policy.PolicyPool([policy.random_weights(num_outputs=A, seed=500 + k) for k in range(R * N)])
    msets = _sets(N, A, R * N, seed=600)
    moa = policy.MOAPool(msets, N)
    pool.seed_sampling(42)
    obs = env.reset()
    h, c = pool.initial_state(m)
    hm, cm = moa.initial_state(m)
    seen, outs = [], []
    for _ in range(6):
        x = pool.features(obs, ids)
        st = pool.policy_step(obs, ids, h, c, features=x)
        s = moa.step(x, ids, st.actions.view(B, N), st.logits, hm, cm)
        seen.append((obs.reshape(-1, 15, 15, 3).clone(), st.actions.clone(), st.logits.clone()))
        outs.append(_rows(moa, s, m))
        h, c, hm, cm = st.h, st.c, s.h, s.c
        obs, _ = env.step(st.actions.view(B, N))
    torch.cuda.synchronize()
    env.close()
    ref = RowwiseReference(msets, N)
    hr, cr = torch.zeros((m, 128), device="cuda"), torch.zeros((m, 128), device="cuda")
    for t, (o, acts, logits) in enumerate(seen):
        x = pool.features(o, ids.reshape(-1))
        want = ref.step(x, ids, acts.view(B, N), logits, hr, cr)
        for name, g, w in zip(NAMES, outs[t], want):
            assert torch.equal(g, w), (t, name)
        hr, cr = want[3], want[4]
    assert len(torch.unique(torch.stack([s[1] for s in seen]))) > 1
    assert float(outs[-1][1].abs().max()) > 0.0
    ref.close()
    pool.close()
    moa.close()


def _policies():
    policy = _policy()
    A, N = 8, 5
    return {"shared": policy.ConvToFCNet(policy.random_weights(num_outputs=A, seed=1)),
            "per_agent": policy.ConvToFCNet([policy.random_weights(num_outputs=A, seed=10 + k) for k in range(N)]),
            "pool": policy.PolicyPool([policy.random_weights(num_outputs=A, seed=20 + k) for k in range(3)])}


@pytest.mark.parametrize("mode", ["sample", "greedy", "given"])
@pytest.mark.parametrize("kind", ["shared", "per_agent", "pool"])
def test_policy_step_with_features_is_bitwise_the_same(kind, mode):
    net = _policies()[kind]
    B, N, A = 260, 5, 8
    m = B * N
    g = torch.Generator(device="cuda").manual_seed(4)
    obs = torch.randint(0, 256, (B, N, 15, 15, 3), dtype=torch.uint8, device="cuda", generator=g)
    ids = torch.randint(0, 4, (B, N), dtype=torch.uint8, device="cuda", generator=g)   # id 3 >= K = 3: skipped agents
    given = torch.randint(-1, A, (m,), dtype=torch.int8, device="cuda", generator=g) if mode == "given" else None
    pool = kind == "pool"
    h, c = net.initial_state(m)
    h = net.state_from_rows(torch.rand((m, 128), device="cuda", generator=g))
    x = net.features(obs, ids) if pool else net.features(obs)
    lead = (obs, ids) if pool else (obs,)
    live = ids.reshape(-1).long() < 3 if pool else torch.ones(m, dtype=torch.bool, device="cuda")
    for t in range(3):
        net.seed_sampling(9 + t)
        a = net.policy_step(*lead, h, c, mode=mode, actions=given)
        counter = net._sample_counter
        assert counter == (1 if mode == "sample" else 0)
        net.seed_sampling(9 + t)
        b = net.policy_step(*lead, h, c, mode=mode, actions=given, features=x)
        assert net._sample_counter == counter   # the same counter advance
        net.seed_sampling(9 + t)
        d = net.policy_step(None, *lead[1:], h, c, mode=mode, actions=given, features=x)   # obs may be None
        for s in (b, d):
            assert torch.equal(s.actions, a.actions)   # a pool's skipped agents: -1 in both, or the given action
            for f in ("logp", "entropy", "logits", "value"):   # bit patterns: logp is NaN where a given action is -1
                assert torch.equal(getattr(s, f)[live].view(torch.int32), getattr(a, f)[live].view(torch.int32)), (t, f)
            assert torch.equal(net.state_rows(s.h, m)[live], net.state_rows(a.h, m)[live])
            assert torch.equal(net.state_rows(s.c, m)[live], net.state_rows(a.c, m)[live])
        h, c = a.h, a.c
    for bad in (x.double(), x.cpu(), x[:-N], x[:, :16]):
        with pytest.raises(ValueError):
            net.policy_step(*lead, h, c, mode=mode, actions=given, features=bad)
    net.close()


def test_errors():
    policy = _policy()
    from sequential_social_dilemma_games_b200 import _lib
    L = _lib.lib
    n, a, B, K = 5, 8, 4, 3
    m = B * n
    sets = _sets(n, a, K, seed=0)
    pool = policy.MOAPool(sets, n)
    moa = policy.MOANet(sets[0], n)
    pnet = policy.ConvToFCNet(policy.random_weights(num_outputs=a, seed=0))
    ppool = policy.PolicyPool([policy.random_weights(num_outputs=a, seed=0)] * 2)
    p = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    x = torch.zeros((m, 32), device="cuda")
    ids = torch.zeros((m,), dtype=torch.uint8, device="cuda")
    joint = torch.zeros((m,), dtype=torch.int8, device="cuda")
    pl = torch.zeros((m, a), device="cuda")
    h, c = pool.initial_state(m)
    hn, cn = torch.empty_like(h), torch.empty_like(c)
    pred, cf = torch.empty((m, n - 1, a), device="cuda"), torch.empty((m, a, n - 1, a), device="cuda")
    ipa, infl = torch.empty((m, n - 1), device="cuda"), torch.empty((m,), device="cuda")
    io = [p(x), p(ids), p(joint), p(pl), p(h), p(c), p(hn), p(cn), p(pred), p(cf), p(ipa), p(infl)]
    step = lambda hd, *, mm=m, div=0, clip=math.inf, args=io: L.ssd_moa_pool_step(hd, *args, mm, div, clip, st)
    assert step(pool._h) == 0 and step(pool._h, div=1) == 0 and step(pool._h, mm=0) == 0
    args = list(io)
    args[9] = None
    assert step(pool._h, args=args) == 0   # counterfactual optional
    for k in range(12):
        if k == 9:
            continue
        args = list(io)
        args[k] = None
        assert step(pool._h, args=args) == -1, k
    assert step(None) == -1
    assert step(pool._h, mm=m - 1) == -1 and b"multiple" in L.ssd_last_error()
    assert step(pool._h, mm=-5) == -1
    for div in (-1, 2):
        assert step(pool._h, div=div) == -1 and b"divergence" in L.ssd_last_error()
    for clip in (math.nan, -1.0):
        assert step(pool._h, clip=clip) == -1 and b"clip" in L.ssd_last_error()
    args = list(io)
    args[0] = C.c_void_p(x.data_ptr() + 4)
    assert step(pool._h, args=args) == -1 and b"aligned" in L.ssd_last_error()
    args = list(io)
    args[6], args[7] = args[4], args[5]
    assert step(pool._h, args=args) == -1 and b"alias" in L.ssd_last_error()
    # handle crossing: the MOA pool step takes no other handle ...
    for other in (moa, pnet, ppool):
        assert step(other._h) == -1 and b"not an MOA pool handle" in L.ssd_last_error()
    # ... the plain MOA step no MOA pool ...
    plain = [io[0]] + io[2:]
    assert L.ssd_moa_step(pool._h, *plain, m, 0, math.inf, st) == -1 and b"ssd_moa_pool_step" in L.ssd_last_error()
    assert L.ssd_moa_step(moa._h, *plain, m, 0, math.inf, st) == 0
    # ... and no policy entry point an MOA pool
    lg, vl = torch.zeros((m, a), device="cuda"), torch.zeros((m,), device="cuda")
    obs = torch.zeros((m, 15, 15, 3), dtype=torch.uint8, device="cuda")
    assert L.ssd_policy_features(pool._h, p(obs), m, p(x), st) == -1 and b"MOA pool" in L.ssd_last_error()
    assert L.ssd_policy_lstm_heads(pool._h, p(x), p(h), p(c), p(hn), p(cn), p(lg), p(vl), None, m, 0, 0, st) == -1
    assert b"MOA pool" in L.ssd_last_error()
    assert L.ssd_policy_lstm_heads_dist(pool._h, p(x), p(h), p(c), p(hn), p(cn), p(lg), p(vl), 0, p(joint), None, None, m, 0, 0, st) == -1
    assert L.ssd_policy_pool_features(pool._h, p(obs), p(ids), m, p(x), st) == -1 and b"pool" in L.ssd_last_error()
    assert L.ssd_policy_pool_lstm_heads(pool._h, p(x), p(ids), p(h), p(c), p(hn), p(cn), p(lg), p(vl), None, m, 0, 0, st) == -1
    assert L.ssd_policy_pool_lstm_heads_dist(pool._h, p(x), p(ids), p(h), p(c), p(hn), p(cn), p(lg), p(vl), 0, p(joint), None, None, m, 0, 0,
                                             st) == -1
    z = np.zeros(4096, np.float32)
    zp = z.ctypes.data_as(C.c_void_p)
    assert L.ssd_policy_set_head_n(pool._h, 3, 128, a, zp, zp, zp, zp, zp, zp, zp) == -1
    # creation: K, null pointers; nothing is allocated
    big = np.zeros(256 * ((32 + 5 * 8) * 512 + 128 * 512 + 512 + 128 * 32 + 32), np.float32)
    bp = big.ctypes.data_as(C.c_void_p)
    out = C.c_void_p()
    for KK in (0, 256):
        assert L.ssd_moa_create_pool(0, KK, n, a, bp, bp, bp, bp, bp, C.byref(out)) == -1 and not out.value
    assert L.ssd_moa_create_pool(0, 3, n, a, bp, None, bp, bp, bp, C.byref(out)) == -1 and not out.value
    assert L.ssd_moa_create_pool(0, 255, n, a, bp, bp, bp, bp, bp, C.byref(out)) == 0 and out.value
    L.ssd_moa_destroy(out)
    torch.cuda.synchronize()
    # Python: ids of the wrong dtype, shape or device; the MOANet checks
    good = ids.reshape(B, n)
    assert pool.step(x, good, joint, pl, h, c).pred.shape == (m, n - 1, a)
    for bad in (good.long(), good.reshape(n, B), good[:3], good.cpu(), good.tolist()):
        with pytest.raises(ValueError):
            pool.step(x, bad, joint, pl, h, c)
    for kw in ({"divergence": "KL"}, {"clip": float("nan")}, {"clip": -1.0}):
        with pytest.raises(ValueError):
            pool.step(x, good, joint, pl, h, c, **kw)
    with pytest.raises(ValueError):
        pool.step(x, good, joint, pl[:, :5], h, c)
    with pytest.raises(ValueError):
        pool.step(x[:7], good, joint, pl, h, c)
    with pytest.raises(ValueError):
        pool.step(x, good, joint, pl, *moa.initial_state(2 * 128 * n))   # not the tiled state of m agents
    with pytest.raises(ValueError):
        policy.MOAPool([], n)
    with pytest.raises(ValueError):
        policy.MOAPool([sets[0], _weights(n, 9, seed=1)], n)
    with pytest.raises(_lib.SsdError):
        policy.MOAPool([sets[0]] * 256, n)
    pool.close()
    moa.close()
    pnet.close()
    ppool.close()
