"""policy_step / ssd_policy_lstm_heads_dist / ssd_policy_pool_lstm_heads_dist: the action of a mode (sampled, greedy or given),
its log-probability and the entropy of the policy, from the fused head kernel.

  sample == act     mode 'sample' draws bitwise what `act` draws and advances the same counter: actions, logits, value, h'
                    and c' over three recurrent steps with act / policy_step calls interleaved (and greedy / given calls in
                    between, which advance nothing), shared, per-agent and pool networks; the pool's skipped agents keep the
                    sentinels of their output rows, logp and entropy included;
  greedy            the first argmax of the returned logits, exactly, constructed ties included;
  logp, entropy     within 2e-6 of float64 computed from the kernel's own returned logits, 1 / 8 / 9 / 15 outputs, every mode;
                    the float64 oracle (oracle/policy_ref.py) bounds logits / value / h / c as in test_policy_gpu.py;
  given             random int8 and uint8 actions, NaN for -1, A and 255; the actions buffer holds what it held (a
                    kernel that wrote back the value it read would pass this check: it sees content only);
  Philox            with all logits 0 the sampled action is the first argmax of the top 24 bits of the words of
                    oracle/philox_ref.py, logp = -log A and entropy = log A;
  unfused route     (cell size 64) the same API in torch, against float64;
  errors            the C ABI's argument checks, handle crossing included, and the Python wrapper's."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from test_policy_gpu import FWD_TOL

pytestmark = pytest.mark.gpu

DIST_TOL = 2e-6   # logp / entropy vs float64 from the kernel's own logits (accurate expf / logf, <= 15 terms)
GA = 128
SEED = 2 ** 64 - 5


def _policy():
    from sequential_social_dilemma_games_b200 import policy
    return policy


def _lib():
    from sequential_social_dilemma_games_b200 import _lib
    return _lib


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _obs(m, seed, steps=3):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randint(0, 256, (m, 15, 15, 3), dtype=torch.uint8, device="cuda", generator=g) for _ in range(steps)]


def _sets(n, A, seed):
    return [_policy().random_weights(num_outputs=A, seed=seed + k) for k in range(n)]


def _net(kind, A, m, seed=40, sets=None):
    """(net, args) of one kind: args(obs) -> the positional arguments before (h, c); pool ids have ~1 % skipped agents."""
    policy = _policy()
    n_sets = {"shared": 1, "per_agent": 5, "pool3": 3, "pool40": 40}[kind]
    sets = sets or _sets(n_sets, A, seed)
    if kind == "shared":
        return policy.ConvToFCNet(sets[0]), lambda o: (o,)
    if kind == "per_agent":
        return policy.ConvToFCNet(sets), lambda o: (o.reshape(-1, 5, 15, 15, 3),)
    g = torch.Generator(device="cuda").manual_seed(seed)
    ids = torch.randint(0, n_sets, (m,), dtype=torch.uint8, device="cuda", generator=g)
    skip = torch.rand((m,), device="cuda", generator=g) < 0.01
    ids[skip] = torch.randint(n_sets, 256, (int(skip.sum()),), dtype=torch.uint8, device="cuda", generator=g)
    return policy.PolicyPool(sets), lambda o: (o, ids)


def _live(net, args, m):
    if not isinstance(net, _policy().PolicyPool):
        return torch.ones((m,), dtype=torch.bool, device="cuda")
    return args(None)[1].long() < net.num_policies


def _dist64(logits, actions):
    """float64 (logp, entropy) from fp32 logits [M, A] and int actions [M] (NaN outside 0..A-1)."""
    l = logits.double()
    ls = torch.log_softmax(l, dim=1)
    a = actions.long()
    ok = (a >= 0) & (a < l.shape[1])
    logp = ls.gather(1, torch.where(ok, a, 0)[:, None]).squeeze(1).masked_fill(~ok, float("nan"))
    return logp, -(ls.exp() * ls).sum(dim=1)


def _check_dist(step, live, actions=None):
    """logp / entropy of a PolicyStep vs float64 from its own logits, on the live rows."""
    a = step.actions if actions is None else actions
    logp64, ent64 = _dist64(step.logits[live], a[live])
    logp, ent = step.logp[live].double(), step.entropy[live].double()
    assert torch.equal(torch.isnan(logp), torch.isnan(logp64))
    ok = ~torch.isnan(logp64)
    if bool(ok.any()):
        assert (logp[ok] - logp64[ok]).abs().max().item() < DIST_TOL
    assert (ent - ent64).abs().max().item() < DIST_TOL
    return logp, ent


# ---------------------------------------------------------------------------------------------------- sample == act
M_SCALE = "4*sms*128+77"


def _m(m):
    return 4 * _sms() * GA + 77 if m == M_SCALE else m


@pytest.mark.parametrize("kind,M", [("shared", 1), ("shared", 127), ("shared", 128), ("shared", 129), ("shared", M_SCALE),
                                    ("per_agent", 5 * 1000), ("per_agent", 5 * (4 * 29 * GA + 77)),
                                    ("pool3", 5123), ("pool3", M_SCALE), ("pool40", 5123), ("pool40", M_SCALE)])
def test_sample_mode_equals_act(kind, M):
    """Three recurrent steps: the reference calls forward + act; the run under test calls greedy and given policy_steps (which
    must not move the counter), then policy_step 'sample' at steps 0 and 2 and act at step 1.  Bitwise on the live rows;
    actions on all rows (-1 for skipped pool agents)."""
    m = _m(M)
    net, args = _net(kind, 8, m)
    live = _live(net, args, m)
    if kind.startswith("pool") and m > 5000:
        assert 0.005 < 1 - live.float().mean().item() < 0.02
    steps = _obs(m, seed=m)
    rows = lambda s: net.state_rows(s, m)
    net.seed_sampling(SEED)
    h, c = net.initial_state(m)
    want = []
    for obs in steps:
        lg, v, h2, c2 = net.forward(*args(obs), h, c)
        a, v_act, h, c = net.act(*args(obs), h, c)
        assert torch.equal(v_act[live], v[live]) and torch.equal(rows(h)[live], rows(h2)[live])
        want.append((a, lg, v, rows(h2), rows(c2)))
    net.seed_sampling(SEED)
    h, c = net.initial_state(m)
    for t, obs in enumerate(steps):
        wa, wl, wv, wh, wc = want[t]
        g = net.policy_step(*args(obs), h, c, mode="greedy")
        given = net.policy_step(*args(obs), h, c, mode="given", actions=g.actions)
        for s in (g, given):   # logits, value, h', c' as the plain head writes them, in every mode
            assert torch.equal(s.logits[live], wl[live]) and torch.equal(s.value[live], wv[live])
            assert torch.equal(rows(s.h)[live], wh[live]) and torch.equal(rows(s.c)[live], wc[live])
        assert torch.equal(given.logp[live], g.logp[live]) and torch.equal(given.entropy[live], g.entropy[live])
        if t == 1:
            a, v, h, c = net.act(*args(obs), h, c)
            assert torch.equal(a, wa) and torch.equal(v[live], wv[live])
        else:
            s = net.policy_step(*args(obs), h, c)
            assert torch.equal(s.actions, wa), t
            assert torch.equal(s.logits[live], wl[live]) and torch.equal(s.value[live], wv[live])
            _check_dist(s, live)
            h, c = s.h, s.c
        assert torch.equal(rows(h)[live], wh[live]) and torch.equal(rows(c)[live], wc[live])
        if not bool(live.all()):
            assert bool((g.actions[~live] == -1).all())
    assert len(torch.unique(want[0][0][live])) > 1 or m < 8
    net.close()


@pytest.mark.parametrize("mode", ["sample", "greedy", "given"])
@pytest.mark.parametrize("K", [3, 40])
def test_pool_skipped_agents_keep_their_sentinels(K, mode):
    """C level, 1 % of the ids >= K: the rows of skipped agents keep the sentinels of every output, logp and entropy included;
    the live rows equal those of a call in which every agent has a pool policy."""
    L = _lib().lib
    m = 4 * _sms() * GA + 77
    pool, args = _net("pool%d" % K, 8, m)
    ids = args(None)[1]
    skip = ids.long() >= K
    assert 0 < int(skip.sum())
    obs = _obs(m, seed=K, steps=1)[0]
    feats = pool.features(obs, ids)
    g = torch.Generator(device="cuda").manual_seed(K)
    h = pool.state_from_rows(torch.rand((m, 128), device="cuda", generator=g) * 2 - 1)
    c = pool.state_from_rows(torch.rand((m, 128), device="cuda", generator=g) * 6 - 3)
    code = _lib().ACT_SAMPLE if mode == "sample" else _lib().ACT_GREEDY if mode == "greedy" else _lib().ACT_GIVEN
    p = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def run(ids_):
        out = (torch.full_like(h, 3.25), torch.full_like(c, -3.25), torch.full((m, 8), 9.5, device="cuda"), torch.full((m,), -9.5, device="cuda"),
               torch.randint(-1, 9, (m,), dtype=torch.int8, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3)),
               torch.full((m,), 1.5, device="cuda"), torch.full((m,), -1.5, device="cuda"))
        a_in = out[4].clone()
        hn, cn, lg, vl, ac, lp, en = out
        assert L.ssd_policy_pool_lstm_heads_dist(pool._h, p(feats), p(ids_), p(h), p(c), p(hn), p(cn), p(lg), p(vl), code, p(ac), p(lp), p(en),
                                                 m, 5, 6, st) == 0
        torch.cuda.synchronize()
        return out, a_in

    (hn, cn, lg, vl, ac, lp, en), a_in = run(ids)
    rows = lambda s: pool.state_rows(s, m)
    assert bool((lg[skip] == 9.5).all()) and bool((vl[skip] == -9.5).all())
    assert bool((rows(hn)[skip] == 3.25).all()) and bool((rows(cn)[skip] == -3.25).all())
    assert bool((lp[skip] == 1.5).all()) and bool((en[skip] == -1.5).all())
    assert torch.equal(ac[skip], a_in[skip])
    if mode == "given":
        assert torch.equal(ac, a_in)
    else:
        assert bool((ac[~skip] >= 0).all()) and bool((ac[~skip] < 8).all())
    full = torch.where(skip, torch.zeros_like(ids), ids)
    feats_full = pool.features(obs, full)
    assert torch.equal(feats_full[~skip], feats[~skip])
    feats.copy_(feats_full)
    (hn2, cn2, lg2, vl2, ac2, lp2, en2), _ = run(full)
    live = ~skip
    for x, y in ((lg, lg2), (vl, vl2), (rows(hn), rows(hn2)), (rows(cn), rows(cn2)), (ac, ac2), (lp, lp2), (en, en2)):
        bits = lambda t: t[live].view(torch.int32) if t.dtype == torch.float32 else t[live]   # logp NaN for invalid given actions
        assert torch.equal(bits(x), bits(y))
    pool.close()


# ---------------------------------------------------------------------------------------------------- greedy, logp, entropy
@pytest.mark.parametrize("A", [1, 8, 9, 15])
@pytest.mark.parametrize("kind", ["shared", "per_agent", "pool3"])
def test_modes_against_float64_from_returned_logits(kind, A):
    """Greedy == np.argmax of the returned logits; logp / entropy of every mode within DIST_TOL of float64; given: random
    actions, -1 and A (NaN), buffer untouched.  With one output logp = entropy = 0 exactly."""
    m = 5 * 2000
    net, args = _net(kind, A, m, seed=60 + A)
    live = _live(net, args, m)
    net.seed_sampling(11)
    h, c = net.initial_state(m)
    g = torch.Generator(device="cuda").manual_seed(A)
    for t, obs in enumerate(_obs(m, seed=A)):
        gr = net.policy_step(*args(obs), h, c, mode="greedy")
        lg = gr.logits[live].cpu().numpy()
        assert np.array_equal(gr.actions[live].long().cpu().numpy(), np.argmax(lg, axis=1))
        _check_dist(gr, live)
        given = torch.randint(-1, A + 1, (m,), dtype=torch.int8, device="cuda", generator=g)
        given[:3] = torch.tensor([-1, A, 0], dtype=torch.int8)
        before = given.clone()
        gv = net.policy_step(*args(obs), h, c, mode="given", actions=given)
        assert gv.actions.data_ptr() == given.data_ptr() and torch.equal(given, before)
        logp, _ = _check_dist(gv, live, given)
        bad = ((given < 0) | (given >= A))[live]
        assert bool(torch.isnan(logp[bad]).all()) and not bool(torch.isnan(logp[~bad]).any())
        # uint8 actions, as stored trajectories often hold them: valid ones are scored, A and above (255 included) get NaN
        u8 = torch.randint(0, A + 2, (m,), dtype=torch.uint8, device="cuda", generator=g)
        u8[:3] = torch.tensor([255, A, 0], dtype=torch.uint8)
        gu = net.policy_step(*args(obs), h, c, mode="given", actions=u8)
        assert torch.equal(gu.actions, torch.where(u8 < A, u8, A).to(torch.int8))
        logp_u, _ = _check_dist(gu, live, u8)
        assert torch.equal(torch.isnan(logp_u), (u8 >= A)[live])
        same = (u8.long() == given.long())[live] & ~torch.isnan(logp_u)
        assert torch.equal(logp_u[same], logp[same])
        sm = net.policy_step(*args(obs), h, c)
        assert bool((sm.actions[live] >= 0).all()) and bool((sm.actions[live] < A).all())
        _check_dist(sm, live)
        for s in (gr, gv, sm):
            assert torch.equal(s.logits[live], gr.logits[live]) and torch.equal(s.value[live], gr.value[live])
        if A == 1:
            for s in (gr, sm):
                assert bool((s.logp[live] == 0).all()) and bool((s.entropy[live] == 0).all())
            assert bool((gv.logp[live][~bad] == 0).all())
        else:
            assert bool((sm.entropy[live] > 0).all()) and bool((sm.logp[live] < 0).all())
        h, c = sm.h, sm.c
    net.close()


@pytest.mark.parametrize("kind", ["shared", "per_agent", "pool3"])
def test_greedy_ties_take_the_first_index(kind):
    """logits_w = 0 and tied biases: every logit row is exactly the bias vector, whose maximum 1.25 sits at 2, 5 and 11."""
    A = 12
    bias = np.array([0, 1, 1.25, -1, 0.5, 1.25, 1, 0, -2, 1, 0.25, 1.25], np.float32)
    sets = _sets(5, A, seed=70)
    for w in sets:
        w["logits_w"][:] = 0
        w["logits_b"] = bias.copy()
    m = 5 * 700
    net, args = _net(kind, A, m, sets=sets[:{"shared": 1, "per_agent": 5, "pool3": 3}[kind]])
    live = _live(net, args, m)
    s = net.policy_step(*args(_obs(m, seed=7, steps=1)[0]), *net.initial_state(m), mode="greedy")
    assert torch.equal(s.logits[live], torch.from_numpy(bias).cuda().expand(int(live.sum()), A))
    assert bool((s.actions[live] == 2).all()) and int(np.argmax(bias)) == 2
    want = float(1.25 - np.log(np.exp(bias.astype(np.float64)).sum()))
    assert (s.logp[live].double() - want).abs().max().item() < DIST_TOL
    net.close()


def test_float64_oracle_bounds_the_fused_route():
    """logits / value / h / c of policy_step within FWD_TOL of oracle/policy_ref.py over three steps."""
    from oracle import policy_ref
    policy = _policy()
    m, A = 600, 9
    w = policy.random_weights(num_outputs=A, seed=80)
    net = policy.ConvToFCNet(w)
    h, c = net.initial_state(m)
    h64, c64 = np.zeros((m, 128)), np.zeros((m, 128))
    for t, obs in enumerate(_obs(m, seed=80)):
        s = net.policy_step(obs, h, c, mode="greedy" if t % 2 else "sample")
        l64, v64, h64, c64 = policy_ref.forward(w, obs.cpu().numpy(), h64, c64)
        for got, want in ((s.logits, l64), (s.value, v64), (net.state_rows(s.h, m), h64), (net.state_rows(s.c, m), c64)):
            assert np.abs(got.cpu().numpy().astype(np.float64) - want).max() < FWD_TOL, t
        _check_dist(s, torch.ones((m,), dtype=torch.bool, device="cuda"))
        h, c = s.h, s.c
    net.close()


def test_sample_mode_follows_philox_words():
    """All logits 0: the action is the first argmax over a of the top 24 bits of word a & 3 of the Philox4x32-10 block
    (m lo, m hi, counter, a >> 2) under key (seed lo, seed hi), from oracle/philox_ref.py; logp = -log A, entropy = log A.
    Agents whose two largest 24-bit values differ by less than 2^12 (the kernel's fast logarithm may order them either way)
    are left out."""
    from oracle import philox_ref
    policy = _policy()
    A, m = 8, 300
    w = policy.random_weights(num_outputs=A, seed=90)
    w["logits_w"][:] = 0
    w["logits_b"][:] = 0
    net = policy.ConvToFCNet(w)
    net.seed_sampling(SEED)
    h, c = net.initial_state(m)
    checked = 0
    for counter, obs in enumerate(_obs(m, seed=90, steps=2)):
        s = net.policy_step(obs, h, c)
        a = s.actions.long().cpu().numpy()
        for i in range(m):
            words = []
            for b in range((A + 3) // 4):
                words += philox_ref.philox4x32_10((i & 0xFFFFFFFF, i >> 32, counter, b), (SEED & 0xFFFFFFFF, SEED >> 32))
            k = np.array(words[:A], np.int64) >> 8
            top = np.sort(k)[-2:]
            if top[1] - top[0] >= 2 ** 12:
                assert a[i] == int(np.argmax(k)), (counter, i)
                checked += 1
        assert (s.logp.double() + math.log(A)).abs().max().item() < DIST_TOL
        assert (s.entropy.double() - math.log(A)).abs().max().item() < DIST_TOL
        h, c = s.h, s.c
    assert checked > 0.9 * 2 * m
    net.close()


# ---------------------------------------------------------------------------------------------------- unfused route
def test_unfused_route_matches_float64():
    """cell size 64 (torch GEMMs around ssd_policy_lstm_cell): the same PolicyStep, float64-bounded; 'sample' with a generator
    draws what `act` draws with the same generator."""
    from oracle import policy_ref
    policy = _policy()
    m, A = 700, 8
    w = policy.random_weights(num_outputs=A, cell_size=64, seed=95)
    net = policy.ConvToFCNet(w)
    assert not net._fused_head
    live = torch.ones((m,), dtype=torch.bool, device="cuda")
    h, c = net.initial_state(m)
    h64, c64 = np.zeros((m, 64)), np.zeros((m, 64))
    for t, obs in enumerate(_obs(m, seed=95)):
        l64, v64, h64, c64 = policy_ref.forward(w, obs.cpu().numpy(), h64, c64)
        gr = net.policy_step(obs, h, c, mode="greedy")
        for got, want in ((gr.logits, l64), (gr.value, v64), (gr.h, h64), (gr.c, c64)):
            assert np.abs(got.cpu().numpy().astype(np.float64) - want).max() < FWD_TOL, t
        assert gr.actions.dtype == torch.int8
        assert np.array_equal(gr.actions.long().cpu().numpy(), np.argmax(gr.logits.cpu().numpy(), axis=1))
        _check_dist(gr, live)
        given = torch.randint(-1, A + 1, (m,), device="cuda", generator=torch.Generator(device="cuda").manual_seed(t))
        gv = net.policy_step(obs, h, c, mode="given", actions=given)
        logp, _ = _check_dist(gv, live, given)
        assert torch.equal(torch.isnan(logp), ((given < 0) | (given >= A)))
        assert torch.equal(gv.actions, given.to(torch.int8))
        u8 = torch.randint(0, A + 2, (m,), dtype=torch.uint8, device="cuda", generator=torch.Generator(device="cuda").manual_seed(t))
        u8[:2] = torch.tensor([255, A], dtype=torch.uint8)
        gu = net.policy_step(obs, h, c, mode="given", actions=u8)
        logp_u, _ = _check_dist(gu, live, u8)
        assert torch.equal(torch.isnan(logp_u), u8 >= A) and torch.equal(gu.actions, torch.where(u8 < A, u8, A).to(torch.int8))
        a_act, _, _, _ = net.act(obs, h, c, generator=torch.Generator(device="cuda").manual_seed(t))
        sm = net.policy_step(obs, h, c, generator=torch.Generator(device="cuda").manual_seed(t))
        assert torch.equal(sm.actions, a_act)
        _check_dist(sm, live)
        h, c = gr.h, gr.c
    net.close()


# ---------------------------------------------------------------------------------------------------- errors
def test_errors():
    policy, _l = _policy(), _lib()
    L = _l.lib
    A, m = 8, 20
    w = policy.random_weights(num_outputs=A, seed=0)
    net, per, pool = policy.ConvToFCNet(w), policy.ConvToFCNet([w] * 5), policy.PolicyPool([w, w])
    p = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    obs = torch.zeros((m, 15, 15, 3), dtype=torch.uint8, device="cuda")
    ids = torch.zeros((m,), dtype=torch.uint8, device="cuda")
    feats = net.features(obs)
    h, c = net.initial_state(m)
    hn, cn = torch.empty_like(h), torch.empty_like(c)
    lg, vl = torch.zeros((m, A), device="cuda"), torch.zeros((m,), device="cuda")
    ac = torch.zeros((m,), dtype=torch.int8, device="cuda")
    lp, en = torch.zeros((m,), device="cuda"), torch.zeros((m,), device="cuda")
    io = [p(feats), p(h), p(c), p(hn), p(cn), p(lg), p(vl)]
    heads = lambda hd, mode, a, n=m: L.ssd_policy_lstm_heads_dist(hd, *io, mode, a, p(lp), p(en), n, 0, 0, st)
    pool_heads = lambda hd, mode, a, n=m: L.ssd_policy_pool_lstm_heads_dist(hd, io[0], p(ids), *io[1:], mode, a, p(lp), p(en), n, 0, 0, st)
    for mode in (0, 1, 2):
        assert heads(net._h, mode, p(ac)) == 0 and pool_heads(pool._h, mode, p(ac)) == 0
        assert L.ssd_policy_lstm_heads_dist(net._h, *io, mode, p(ac), None, None, m, 0, 0, st) == 0   # logp, entropy optional
    for mode in (-1, 3, 100):
        assert heads(net._h, mode, p(ac)) == -1 and b"mode" in L.ssd_last_error()
        assert pool_heads(pool._h, mode, p(ac)) == -1 and b"mode" in L.ssd_last_error()
    for mode in (0, 1, 2):
        assert heads(net._h, mode, None) == -1 and b"actions" in L.ssd_last_error()
        assert pool_heads(pool._h, mode, None) == -1 and b"actions" in L.ssd_last_error()
    assert heads(pool._h, 0, p(ac)) == -1 and b"pool" in L.ssd_last_error()                  # handle crossing, both ways
    assert pool_heads(net._h, 0, p(ac)) == -1 and b"pool" in L.ssd_last_error()
    assert pool_heads(per._h, 0, p(ac)) == -1
    assert heads(None, 0, p(ac)) == -1 and pool_heads(None, 0, p(ac)) == -1
    assert heads(net._h, 0, p(ac), n=-1) == -1 and pool_heads(pool._h, 0, p(ac), n=-1) == -1
    assert L.ssd_policy_lstm_heads_dist(net._h, None, *io[1:], 0, p(ac), p(lp), p(en), m, 0, 0, st) == -1
    assert L.ssd_policy_pool_lstm_heads_dist(pool._h, io[0], None, *io[1:], 0, p(ac), p(lp), p(en), m, 0, 0, st) == -1
    mis = C.c_void_p(feats.data_ptr() + 4)
    assert L.ssd_policy_lstm_heads_dist(net._h, mis, *io[1:], 0, p(ac), p(lp), p(en), m, 0, 0, st) == -1 and b"aligned" in L.ssd_last_error()
    # per-agent handle: the num_agents % P rule of ssd_policy_lstm_heads
    hp, cp = per.initial_state(m)
    io_p = [p(feats), p(hp), p(cp), p(torch.empty_like(hp)), p(torch.empty_like(cp)), p(lg), p(vl)]
    assert L.ssd_policy_lstm_heads_dist(per._h, *io_p, 0, p(ac), p(lp), p(en), m, 0, 0, st) == 0
    assert L.ssd_policy_lstm_heads_dist(per._h, *io_p, 0, p(ac), p(lp), p(en), m - 1, 0, 0, st) == -1 and b"multiple" in L.ssd_last_error()
    assert heads(net._h, 0, p(ac), n=0) == 0 and pool_heads(pool._h, 0, p(ac), n=0) == 0
    torch.cuda.synchronize()
    # Python: the mode, and actions only (and always) in mode 'given'
    for bad in ("Sample", "argmax", 0, None):
        with pytest.raises(ValueError):
            net.policy_step(obs, h, c, mode=bad)
        with pytest.raises(ValueError):
            pool.policy_step(obs, ids, h, c, mode=bad)
    with pytest.raises(ValueError):
        net.policy_step(obs, h, c, actions=ac)
    with pytest.raises(ValueError):
        pool.policy_step(obs, ids, h, c, mode="greedy", actions=ac)
    for bad in (None, ac[:5], ac.float(), ac.bool(), ac.cpu(), ac.tolist()):
        with pytest.raises(ValueError):
            net.policy_step(obs, h, c, mode="given", actions=bad)
        with pytest.raises(ValueError):
            pool.policy_step(obs, ids, h, c, mode="given", actions=bad)
    with pytest.raises(ValueError):
        pool.policy_step(obs, ids.long(), h, c)
    # wider integer actions are checked before the narrowing: 135 is not action 7
    s = net.policy_step(obs, h, c, mode="given", actions=torch.tensor([135, -200, 7] + [0] * (m - 3), device="cuda"))
    assert bool(torch.isnan(s.logp[:2]).all()) and not bool(torch.isnan(s.logp[2:]).any())
    for n in (net, per, pool):
        n.close()
