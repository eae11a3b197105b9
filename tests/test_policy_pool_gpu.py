"""Policy pool (PolicyPool, ssd_policy_create_pool / ssd_policy_pool_features / ssd_policy_pool_lstm_heads): K weight sets,
agent m evaluated with set policy_ids[m] of each call.  Each agent runs the instruction sequence of the shared network on its
set's weights and the sampler is keyed by m, so the reference -- K shared networks, each run on ALL M agents, keeping the
rows whose id is k -- is matched bitwise, actions included; the float64 oracle (oracle/policy_ref.py) bounds the columns to
the tolerances of test_policy_gpu.py."""
import ctypes as C

import numpy as np
import pytest
import torch

from test_policy_gpu import FWD_TOL, TRUNK_TOL

pytestmark = pytest.mark.gpu

NUM_OUTPUTS = 8


def _policy():
    from sequential_social_dilemma_games_b200 import policy
    return policy


def _sets(K, seed=300, num_outputs=NUM_OUTPUTS):
    policy = _policy()
    return [policy.random_weights(num_outputs=num_outputs, seed=seed + k) for k in range(K)]


@pytest.fixture(scope="module")
def env_obs():
    """Three consecutive observation tensors of Harvest (700 envs x 5 agents) and Cleanup (500 envs x 5 agents) from the step
    kernel, flattened to 6 000 agents."""
    from sequential_social_dilemma_games_b200.batched import BatchedSSDEnv, make_config
    out = []
    envs = [BatchedSSDEnv(make_config(game, num_agents=5), B, seed=11) for game, B in (("harvest", 700), ("cleanup", 500))]
    for e in envs:
        e.reset()
    g = torch.Generator(device="cuda").manual_seed(6)
    for _ in range(3):
        obs = []
        for e in envs:
            a = torch.randint(0, NUM_OUTPUTS, (e.num_envs, 5), dtype=torch.int8, device="cuda", generator=g)
            o, _ = e.step(a)
            obs.append(o.reshape(-1, 15, 15, 3))
        out.append(torch.cat(obs))
    torch.cuda.synchronize()
    for e in envs:
        e.close()
    return out


def _obs_steps(source, M, env_obs, seed):
    if source == "env":   # beyond the recorded agents, the recorded observations again
        return [o.repeat((M + o.shape[0] - 1) // o.shape[0], 1, 1, 1)[:M].contiguous() for o in env_obs]
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randint(0, 256, (M, 15, 15, 3), dtype=torch.uint8, device="cuda", generator=g) for _ in range(3)]


class RowwiseReference(object):
    """K shared networks, each evaluated on all M agents; agent m keeps the outputs of network ids[m].  (h, c) are carried
    agent-major in the tiled layout, which the shared network and the pool share."""

    def __init__(self, sets, seed):
        policy = _policy()
        self.nets = [policy.ConvToFCNet(w) for w in sets]
        for n in self.nets:
            n.seed_sampling(seed)

    def step(self, obs, ids, h, c):
        m = obs.shape[0]
        ids = ids.reshape(-1).long()
        out = None
        for k, net in enumerate(self.nets):
            sel = ids == k
            f = net.features(obs)
            lg, v, h2, c2 = net.forward(obs, h, c)
            a, _, _, _ = net.act(obs, h, c)   # every net is asked once per step: its Philox counter stays in step with the pool's
            r = (f, lg, v, net.state_rows(h2, m), net.state_rows(c2, m), a)
            if out is None:
                out = [torch.zeros_like(t) for t in r]
                out[5].fill_(-1)
            for o, t in zip(out, r):
                o[sel] = t[sel]
        f, lg, v, hr, cr, a = out
        return f, lg, v, hr, cr, a

    def close(self):
        for n in self.nets:
            n.close()


def _run_pool(pool, steps, ids_per_step, seed, h=None, c=None):
    m = steps[0].shape[0]
    pool.seed_sampling(seed)
    if h is None:
        h, c = pool.initial_state(m)
    res = []
    for obs, ids in zip(steps, ids_per_step):
        f = pool.features(obs, ids)
        lg, v, h2, c2 = pool.forward(obs, ids, h, c)
        a, v2, h, c = pool.act(obs, ids, h, c)
        live = ids.reshape(-1).long() < pool.num_policies   # the value of a skipped agent is not written
        assert torch.equal(v2[live], v[live])
        res.append((f, lg, v, pool.state_rows(h2, m), pool.state_rows(c2, m), a, h, c))
    return res


def _check_against_reference(sets, steps, ids_per_step, seed=77):
    """Pool vs the row-wise reference over the recurrent steps, bitwise, with the reference's state carried agent-major."""
    policy = _policy()
    m = steps[0].shape[0]
    pool = policy.PolicyPool(sets)
    ref = RowwiseReference(sets, seed)
    got = _run_pool(pool, steps, ids_per_step, seed)
    h, c = pool.initial_state(m)
    for t, (obs, ids) in enumerate(zip(steps, ids_per_step)):
        live = ids.reshape(-1).long() < len(sets)   # the pool writes nothing but action -1 for the other agents
        want = ref.step(obs, ids, h, c)
        for name, g, w in zip(("features", "logits", "value", "h", "c"), got[t][:5], want):
            assert torch.equal(g[live], w[live]), (t, name)
        assert torch.equal(got[t][5], want[5]), (t, "actions")
        h, c = pool.state_from_rows(want[3]), pool.state_from_rows(want[4])
    pool.close()
    ref.close()
    return got


@pytest.mark.parametrize("source", ["random", "env"])
@pytest.mark.parametrize("M", [1, 127, 128, 129, 5123])
def test_pool_of_one_equals_shared_net(M, source, env_obs):
    policy = _policy()
    w = policy.random_weights(num_outputs=NUM_OUTPUTS, seed=21)
    shared, pool = policy.ConvToFCNet(w), policy.PolicyPool([w])
    assert pool.num_policies == 1
    steps = _obs_steps(source, M, env_obs, seed=M)
    ids = torch.zeros((M,), dtype=torch.uint8, device="cuda")
    hs, cs = shared.initial_state(M)
    hp, cp = pool.initial_state(M)
    assert hp.shape == hs.shape
    shared.seed_sampling(99)
    pool.seed_sampling(99)
    for obs in steps:
        assert torch.equal(pool.features(obs, ids), shared.features(obs))
        ls, vs, hs2, cs2 = shared.forward(obs, hs, cs)
        lp, vp, hp2, cp2 = pool.forward(obs, ids, hp, cp)
        assert torch.equal(lp, ls) and torch.equal(vp, vs)
        assert torch.equal(pool.state_rows(hp2, M), shared.state_rows(hs2, M))
        assert torch.equal(pool.state_rows(cp2, M), shared.state_rows(cs2, M))
        a_s, _, hs, cs = shared.act(obs, hs, cs)
        a_p, _, hp, cp = pool.act(obs, ids, hp, cp)
        assert torch.equal(a_p, a_s)
        assert torch.equal(pool.state_rows(hp, M), shared.state_rows(hs, M))
    shared.close()
    pool.close()


@pytest.mark.parametrize("source", ["random", "env"])
@pytest.mark.parametrize("N", [2, 5, 16])
def test_identity_mapping_equals_per_agent_net(N, source, env_obs):
    policy = _policy()
    B = 300
    M = B * N
    sets = _sets(N)
    per, pool = policy.ConvToFCNet(sets), policy.PolicyPool(sets)
    steps = [o.reshape(B, N, 15, 15, 3) for o in _obs_steps(source, M, env_obs, seed=N)]
    ids = torch.arange(N, dtype=torch.uint8, device="cuda").repeat(B, 1)
    hq, cq = per.initial_state(M)
    hp, cp = pool.initial_state(M)
    per.seed_sampling(5)
    pool.seed_sampling(5)
    for obs in steps:
        assert torch.equal(pool.features(obs, ids), per.features(obs))
        lq, vq, hq2, cq2 = per.forward(obs, hq, cq)
        lp, vp, hp2, cp2 = pool.forward(obs, ids, hp, cp)
        assert torch.equal(lp, lq) and torch.equal(vp, vq)
        assert torch.equal(pool.state_rows(hp2, M), per.state_rows(hq2, M))
        assert torch.equal(pool.state_rows(cp2, M), per.state_rows(cq2, M))
        a_q, _, hq, cq = per.act(obs, hq, cq)
        a_p, _, hp, cp = pool.act(obs, ids, hp, cp)
        assert torch.equal(a_p, a_q)
    per.close()
    pool.close()


def _ids_with_sizes(M, K, sizes, seed, skipped=0):
    """uint8 [M]: policy k holds exactly sizes[k] agents for the policies in `sizes`, `skipped` agents have an id >= K, the
    other policies share the rest at random."""
    rng = np.random.RandomState(seed)
    fixed = np.concatenate([np.full(n, k) for k, n in sizes.items()] + [rng.randint(K, 256, skipped)])
    others = np.array([k for k in range(K) if k not in sizes])
    ids = np.concatenate([fixed, rng.choice(others, M - len(fixed))])
    rng.shuffle(ids)
    return torch.from_numpy(ids.astype(np.uint8)).cuda()


SCALE_M = 65536 * 5   # 65 536 Harvest envs x 5 agents: a CTA of the trunk and head runs many tiles, the assignment 80 chunks


@pytest.mark.parametrize("K,sizes,M", [
    pytest.param(3, {0: 129, 1: 0}, 5123, id="3-sizes0"),                               # policy 2 takes the rest
    pytest.param(3, {1: 1, 2: 127}, 5123, id="3-sizes1"),
    pytest.param(40, {0: 0, 1: 1, 2: 127, 3: 128, 4: 129}, 5123, id="40-sizes2"),
    pytest.param(255, {7: 127, 8: 128, 9: 129, 10: 1, 11: 0}, 5123, id="255-sizes3"),
    pytest.param(3, {0: 129, 1: 0}, SCALE_M, id="3-sizes0-M327680"),                     # long same-policy segments
    pytest.param(255, {7: 127, 8: 128, 9: 129, 10: 1, 11: 0}, SCALE_M, id="255-sizes3-M327680"),   # many switches per CTA
])
@pytest.mark.parametrize("source", ["random", "env"])
def test_random_ids_match_rowwise_reference(K, sizes, M, source, env_obs):
    """At 327 680 agents about 1 % of the ids are >= K (skipped)."""
    skipped = M // 100 if M == SCALE_M else 0
    steps = _obs_steps(source, M, env_obs, seed=K)
    ids = _ids_with_sizes(M, K, sizes, seed=K, skipped=skipped)
    counts = torch.bincount(ids.long(), minlength=256).cpu().numpy()
    assert counts[K:].sum() == skipped
    for k, n in sizes.items():
        assert counts[k] == n
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    if M == SCALE_M:   # every CTA of the trunk and the head runs at least four tiles
        assert sum((int(n) + 127) // 128 for n in counts[:K]) >= 4 * sms
    _check_against_reference(_sets(K), steps, [ids] * 3)


@pytest.mark.parametrize("M", [129, 5123])
def test_one_policy_holds_every_agent(M):
    K = 40
    steps = _obs_steps("random", M, None, seed=M)
    _check_against_reference(_sets(K), steps, [torch.full((M,), 17, dtype=torch.uint8, device="cuda")] * 3)


def test_reassignment_between_steps(env_obs):
    """The ids change at every step while (h, c) stay agent-major; the reference carries h and c per agent."""
    K, M = 7, 4000
    g = torch.Generator(device="cuda").manual_seed(1)
    ids = [torch.randint(0, K, (M,), dtype=torch.uint8, device="cuda", generator=g) for _ in range(3)]
    got = _check_against_reference(_sets(K), _obs_steps("env", M, env_obs, 0), ids)
    assert not torch.equal(got[0][5], got[1][5])


def test_skipped_agents_are_not_written():
    policy = _policy()
    from sequential_social_dilemma_games_b200 import _lib
    L = _lib.lib
    K, M = 5, 1000
    sets = _sets(K)
    pool = policy.PolicyPool(sets)
    g = torch.Generator(device="cuda").manual_seed(2)
    obs = torch.randint(0, 256, (M, 15, 15, 3), dtype=torch.uint8, device="cuda", generator=g)
    ids = torch.randint(0, K + 3, (M,), dtype=torch.uint8, device="cuda", generator=g)
    ids[::97] = 255
    skip = ids.long() >= K
    full_ids = torch.where(skip, torch.zeros_like(ids), ids)   # the same agents with a pool policy each
    assert 0 < int(skip.sum()) < M
    # C level: sentinel-filled outputs keep the sentinel in the skipped rows
    p = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    feats = torch.full((M, 32), 7.5, device="cuda")
    assert L.ssd_policy_pool_features(pool._h, p(obs), p(ids), M, p(feats), st) == 0
    h, c = pool.initial_state(M)
    h = pool.state_from_rows(torch.rand((M, 128), device="cuda", generator=g))
    hn, cn = torch.full_like(h, 3.25), torch.full_like(c, -3.25)
    lg, vl = torch.full((M, NUM_OUTPUTS), 9.5, device="cuda"), torch.full((M,), -9.5, device="cuda")
    ac = torch.full((M,), 42, dtype=torch.int8, device="cuda")
    assert L.ssd_policy_pool_lstm_heads(pool._h, p(feats), p(ids), p(h), p(c), p(hn), p(cn), p(lg), p(vl), p(ac), M, 3, 4, st) == 0
    torch.cuda.synchronize()
    assert bool((feats[skip] == 7.5).all()) and bool((lg[skip] == 9.5).all()) and bool((vl[skip] == -9.5).all())
    assert bool((ac[skip] == 42).all()) and bool((ac[~skip] >= 0).all())
    assert bool((pool.state_rows(hn, M)[skip] == 3.25).all()) and bool((pool.state_rows(cn, M)[skip] == -3.25).all())
    # the live agents' outputs equal the run in which every agent has a pool policy
    feats2 = pool.features(obs, full_ids)
    lg2 = torch.empty_like(lg)
    vl2, ac2 = torch.empty_like(vl), torch.empty_like(ac)
    hn2, cn2 = torch.empty_like(h), torch.empty_like(c)
    assert L.ssd_policy_pool_lstm_heads(pool._h, p(feats2), p(full_ids), p(h), p(c), p(hn2), p(cn2), p(lg2), p(vl2), p(ac2), M, 3, 4, st) == 0
    live = ~skip
    assert torch.equal(feats[live], feats2[live]) and torch.equal(lg[live], lg2[live]) and torch.equal(vl[live], vl2[live])
    assert torch.equal(ac[live], ac2[live])
    assert torch.equal(pool.state_rows(hn, M)[live], pool.state_rows(hn2, M)[live])
    assert torch.equal(pool.state_rows(cn, M)[live], pool.state_rows(cn2, M)[live])
    # Python level: act returns -1 for the skipped agents
    pool.seed_sampling(8)
    a, _, _, _ = pool.act(obs, ids, h, c)
    assert bool((a[skip] == -1).all()) and bool((a[live] >= 0).all())
    pool.close()


def test_matches_float64_oracle():
    _check_float64_oracle(NUM_OUTPUTS)


@pytest.mark.parametrize("num_outputs", [1, 15])
def test_matches_float64_oracle_head_widths(num_outputs):
    """The value in head column 1 and 15: the pool head selects it with code of its own."""
    _check_float64_oracle(num_outputs)


def _check_float64_oracle(num_outputs):
    from oracle import policy_ref
    policy = _policy()
    K, M = 3, 600
    sets = _sets(K, num_outputs=num_outputs)
    pool = policy.PolicyPool(sets)
    steps = _obs_steps("random", M, None, seed=12)
    ids = torch.randint(0, K, (M,), dtype=torch.uint8, device="cuda", generator=torch.Generator(device="cuda").manual_seed(12))
    idn = ids.cpu().numpy()
    h, c = pool.initial_state(M)
    h64, c64 = np.zeros((M, 128)), np.zeros((M, 128))
    for t, obs in enumerate(steps):
        f = pool.features(obs, ids).cpu().numpy().astype(np.float64)
        lg, v, h, c = pool.forward(obs, ids, h, c)
        lg, v = lg.cpu().numpy(), v.cpu().numpy()
        hr, cr = pool.state_rows(h, M).cpu().numpy(), pool.state_rows(c, M).cpu().numpy()
        on = obs.cpu().numpy()
        for k in range(K):
            sel = idn == k
            if t == 0:
                assert np.abs(f[sel] - policy_ref.features(sets[k], on[sel])).max() < TRUNK_TOL
            l64, v64, hh, cc = policy_ref.forward(sets[k], on[sel], h64[sel], c64[sel])
            h64[sel], c64[sel] = hh, cc
            for got, want in ((lg[sel], l64), (v[sel], v64), (hr[sel], hh), (cr[sel], cc)):
                assert np.abs(got.astype(np.float64) - want).max() < FWD_TOL, (t, k)
    pool.close()


def test_closed_loop_runs_by_block_mapping():
    """BatchedSSDEnv (300 Harvest envs x 5 agents) -> pool act -> env for six steps; K = 3 runs x 5 agents, env b belongs to
    run b mod 3: ids[b, n] = 5 (b mod 3) + n.  The actions equal the row-wise reference's on the recorded observations."""
    policy = _policy()
    from sequential_social_dilemma_games_b200.batched import BatchedSSDEnv, make_config
    R, N, B = 3, 5, 300
    sets = _sets(R * N, seed=500)
    ids = (N * (torch.arange(B, device="cuda")[:, None] % R) + torch.arange(N, device="cuda")[None, :]).to(torch.uint8)
    env = BatchedSSDEnv(make_config("harvest", num_agents=N), B, seed=5)
    pool = policy.PolicyPool(sets)
    pool.seed_sampling(42)
    obs = env.reset()
    h, c = pool.initial_state(B * N)
    seen, acts = [], []
    for _ in range(6):
        seen.append(obs.reshape(-1, 15, 15, 3).clone())
        a, value, h, c = pool.act(obs, ids, h, c)
        acts.append(a)
        obs, rew = env.step(a.view(B, N))
    torch.cuda.synchronize()
    env.close()
    pool.close()
    ref = RowwiseReference(sets, 42)
    hr, cr = ref.nets[0].initial_state(B * N)
    for t, o in enumerate(seen):
        f, lg, v, h_rows, c_rows, a = ref.step(o, ids, hr, cr)
        assert torch.equal(a, acts[t]), t
        hr, cr = ref.nets[0].state_from_rows(h_rows), ref.nets[0].state_from_rows(c_rows)
    ref.close()
    assert len(torch.unique(torch.stack(acts))) > 1


def test_errors():
    policy = _policy()
    from sequential_social_dilemma_games_b200 import _lib
    L = _lib.lib
    w = policy.random_weights(num_outputs=NUM_OUTPUTS, seed=0)
    with pytest.raises(ValueError):
        policy.PolicyPool([])
    with pytest.raises(_lib.SsdError):
        policy.PolicyPool([w] * 256)
    names = ("conv_w", "conv_b", "fc1_w", "fc1_b", "fc2_w", "fc2_b", "lstm_w", "lstm_u", "lstm_b", "logits_w", "logits_b", "value_w", "value_b")
    arrs = [np.ascontiguousarray(w[k]) for k in names]
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    hh = C.c_void_p()
    for K in (0, 256, -1):
        assert L.ssd_policy_create_pool(7, 0, K, 128, NUM_OUTPUTS, *[ptr(a) for a in arrs], C.byref(hh)) == -1 and not hh.value
    assert L.ssd_policy_create_pool(5, 0, 1, 128, NUM_OUTPUTS, *[ptr(a) for a in arrs], C.byref(hh)) == -3 and not hh.value
    assert b"15x15" in L.ssd_last_error()
    assert L.ssd_policy_create_pool(7, 0, 1, 64, NUM_OUTPUTS, *[ptr(a) for a in arrs], C.byref(hh)) == -3 and not hh.value
    assert L.ssd_policy_create_pool(7, 0, 1, 128, 16, *[ptr(a) for a in arrs], C.byref(hh)) == -3 and not hh.value
    # mismatched weight shapes; a head that is not the fused one
    w9 = policy.random_weights(num_outputs=9, seed=1)
    with pytest.raises(ValueError):
        policy.PolicyPool([w, w9])
    with pytest.raises(ValueError):
        policy.PolicyPool([policy.random_weights(num_outputs=NUM_OUTPUTS, cell_size=64, seed=s) for s in range(2)])
    with pytest.raises(ValueError):
        policy.PolicyPool([{k: v for k, v in w.items() if not k.startswith(("lstm", "logits", "value"))}] * 2)
    # ids of the wrong dtype, shape or device
    pool = policy.PolicyPool([w, w])
    obs = torch.zeros((4, 5, 15, 15, 3), dtype=torch.uint8, device="cuda")
    good = torch.zeros((4, 5), dtype=torch.uint8, device="cuda")
    assert pool.features(obs, good).shape == (20, 32)
    for bad in (good.long(), good.reshape(20), good[:3], good.cpu()):
        with pytest.raises(ValueError):
            pool.features(obs, bad)
        with pytest.raises(ValueError):
            pool.act(obs, bad, *pool.initial_state(20))
    # a pool handle at the other entry points, and the reverse
    net = policy.ConvToFCNet(w)
    p = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    flat = obs.reshape(20, 15, 15, 3)
    ids = good.reshape(20)
    feats = torch.zeros((20, 32), device="cuda")
    h, c = pool.initial_state(20)
    lg, vl = torch.zeros((20, NUM_OUTPUTS), device="cuda"), torch.zeros((20,), device="cuda")
    assert L.ssd_policy_features(pool._h, p(flat), 20, p(feats), st) == -1 and b"pool" in L.ssd_last_error()
    assert L.ssd_policy_lstm_heads(pool._h, p(feats), p(h), p(c), p(h), p(c), p(lg), p(vl), None, 20, 0, 0, st) == -1
    assert L.ssd_policy_set_head_n(pool._h, 2, 128, NUM_OUTPUTS, *[ptr(a) for a in arrs[6:]]) == -1
    assert L.ssd_policy_pool_features(net._h, p(flat), p(ids), 20, p(feats), st) == -1 and b"pool" in L.ssd_last_error()
    assert L.ssd_policy_pool_lstm_heads(net._h, p(feats), p(ids), p(h), p(c), p(h), p(c), p(lg), p(vl), None, 20, 0, 0, st) == -1
    net.close()
    pool.close()
