"""The MOA kernel (csrc/ssd_policy_moa.cu, `policy.MOANet`) against the float64 restatement oracle/moa_ref.py, against its own
returned logits, and against itself across weight maps and batch decompositions.

MOA_TOL: pred, h', c' and the counterfactual logits over three recurrent steps carry the error of the policy head's fused
route (FWD_TOL: fp16 x, h and [Wx; U] in the gate GEMM, tanh.approx in the cell update), and nothing larger: the one-hot rows
and Dense((N-1) A) are fp32.  A logit error e moves each log-probability by at most 2 e, so a divergence term
sum p (log p - log q) moves by about 4 e per other agent to first order; the influence tolerance allows twice that, 8 e per
other agent."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from test_policy_gpu import FWD_TOL

pytestmark = pytest.mark.gpu

MOA_TOL = FWD_TOL
OWN_TOL = 1e-5   # influence vs float64 recomputed from the kernel's own logits (accurate expf / logf in fp32)
# every shape class of the kernel (N = 2..16, A = 1..15, (N - 1) A <= 64)
SHAPE_CLASSES = [(2, 1), (16, 1),           # A = 1: no counterfactual drain on warps 4-7, the influence is exactly 0
                 (2, 15), (5, 15),          # A >= 10
                 (16, 4), (13, 5),          # N >= 10: the pass-0 loop over the others runs past 8
                 (2, 9), (4, 3), (3, 7),    # (N - 1) A not a multiple of 4: a partial last column block of moa_logits_w
                 (8, 9)]                    # (N - 1) A = 63
CASES = [(2, 8), (5, 8), (5, 9), (8, 8), (9, 8)] + SHAPE_CLASSES


def _policy():
    from sequential_social_dilemma_games_b200 import policy
    return policy


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _weights(n, a, seed):
    """random_moa_weights with the own-action rows scaled by 8: random init gives influences of ~1e-4, this ~1e-2."""
    w = _policy().random_moa_weights(n, a, seed=seed)
    w["moa_lstm_w"][32:32 + a] *= 8.0
    return w


def _sets(n, a, count, seed):
    return [_weights(n, a, seed + k) for k in range(count)]


def _inputs(b, n, a, seed, steps=3):
    g = torch.Generator(device="cuda").manual_seed(seed)
    m = b * n
    out = []
    for _ in range(steps):
        x = torch.relu(torch.randn((m, 32), device="cuda", generator=g))
        joint = torch.randint(0, a, (b, n), device="cuda", generator=g).to(torch.int8)
        pl = 2.0 * torch.randn((m, a), device="cuda", generator=g)
        out.append((x, joint, pl))
    return out


def _np(t):
    return t.detach().cpu().numpy().astype(np.float64)


def _oracle_rows(sets, n, x, joint, pl, h, c, a, **kw):
    """moa_ref.moa_forward with weight set m % n for agent m when len(sets) == n."""
    from oracle import moa_ref
    outs = [moa_ref.moa_forward(w, x, joint, pl, h, c, a, **kw) for w in sets]
    if len(outs) == 1:
        return outs[0]
    sel = np.arange(x.shape[0]) % n
    return {k: np.stack([outs[s][k][m] for m, s in enumerate(sel)]) for k in outs[0]}


@pytest.mark.parametrize("kind", ["shared", "per_agent"])
@pytest.mark.parametrize("n,a", CASES)
def test_against_float64_oracle(n, a, kind):
    policy = _policy()
    b = 157   # 157 n agents: two groups per weight set, the second ragged
    sets = _sets(n, a, 1 if kind == "shared" else n, seed=10 * n + a)
    net = policy.MOANet(sets[0] if kind == "shared" else sets, n)
    m = b * n
    h, c = net.initial_state(m)
    g = torch.Generator().manual_seed(n * 100 + a)
    hr = 0.5 * torch.randn((m, 128), generator=g, dtype=torch.float64).numpy()
    cr = 0.5 * torch.randn((m, 128), generator=g, dtype=torch.float64).numpy()
    h, c = net.state_from_rows(torch.from_numpy(hr).float().cuda()), net.state_from_rows(torch.from_numpy(cr).float().cuda())
    hr, cr = _np(net.state_rows(h, m)), _np(net.state_rows(c, m))
    for t, (x, joint, pl) in enumerate(_inputs(b, n, a, seed=n * a)):
        s = net.step(x, joint, pl, h, c, counterfactuals=True)
        ref = _oracle_rows(sets, n, _np(x), _np(joint).astype(np.int64), _np(pl), hr, cr, a)
        tol_infl = 8 * MOA_TOL * (n - 1)
        for name, got, want, tol in (("pred", s.pred, ref["pred"], MOA_TOL), ("h", net.state_rows(s.h, m), ref["h"], MOA_TOL),
                                     ("c", net.state_rows(s.c, m), ref["c"], MOA_TOL),
                                     ("counterfactual", s.counterfactual, ref["counterfactual"], MOA_TOL),
                                     ("influence_per_agent", s.influence_per_agent, ref["influence_per_agent"], tol_infl),
                                     ("influence", s.influence, ref["influence"], tol_infl)):
            err = np.abs(_np(got) - want).max()
            assert err < tol, (t, name, err)
        assert np.abs(ref["pred"]).max() > 0.1   # not vacuous
        if a == 1:   # one action: every softmax is exactly 1, so is every marginal
            assert bool((s.influence == 0).all()) and bool((s.influence_per_agent == 0).all())
        else:
            assert np.abs(ref["influence"]).max() > 1e-3   # not vacuous
        h, c = s.h, s.c
        hr, cr = ref["h"], ref["c"]
    net.close()


@pytest.mark.parametrize("n,a", [(5, 8), (9, 8)])
def test_counterfactual_at_the_actual_action_is_pred(n, a):
    net = _policy().MOANet(_sets(n, a, n, seed=3), n)
    x, joint, pl = _inputs(301, n, a, seed=5, steps=1)[0]
    h, c = net.initial_state(x.shape[0])
    s = net.step(x, joint, pl, h, c, counterfactuals=True)
    idx = joint.reshape(-1).long()
    at = s.counterfactual[torch.arange(x.shape[0], device="cuda"), idx]
    assert torch.equal(at, s.pred)
    s2 = net.step(x, joint, pl, h, c)
    assert s2.counterfactual is None
    m = x.shape[0]
    for got, want in zip(_rows_of(net, s2, m), _rows_of(net, s, m)):   # the state's padding rows are not written
        assert torch.equal(got, want)
    net.close()


@pytest.mark.parametrize("divergence", ["kl", "jsd"])
@pytest.mark.parametrize("n,a", [(2, 8), (5, 9), (9, 8)] + SHAPE_CLASSES)
def test_influence_against_its_own_logits(n, a, divergence):
    from oracle import moa_ref
    net = _policy().MOANet(_sets(n, a, 1, seed=7), n)
    x, joint, pl = _inputs(400, n, a, seed=9, steps=1)[0]
    h, c = net.initial_state(x.shape[0])
    s = net.step(x, joint, pl, h, c, divergence=divergence, counterfactuals=True)
    ipa, infl = moa_ref.influence_from(_np(s.pred), _np(s.counterfactual), _np(pl), _np(joint).astype(np.int64), a, divergence)
    assert np.abs(_np(s.influence_per_agent) - ipa).max() < OWN_TOL
    assert np.abs(_np(s.influence) - infl).max() < OWN_TOL
    if a == 1:   # exactly 0; a clip has nothing to act on
        assert bool((s.influence == 0).all()) and bool((s.influence_per_agent == 0).all())
        net.close()
        return
    clip = float(np.float32(np.median(infl)))   # the C ABI takes clip as a float
    s2 = net.step(x, joint, pl, h, c, divergence=divergence, clip=clip, counterfactuals=True)
    _, infl_c = moa_ref.influence_from(_np(s2.pred), _np(s2.counterfactual), _np(pl), _np(joint).astype(np.int64), a, divergence, clip)
    assert np.abs(_np(s2.influence) - infl_c).max() < OWN_TOL
    assert float(s2.influence.max()) <= clip and (infl > clip).any()
    if divergence == "jsd":
        assert float(s.influence_per_agent.max()) <= math.log(2) + 1e-6
    net.close()


@pytest.mark.parametrize("divergence", ["kl", "jsd"])
@pytest.mark.parametrize("n,a", [(5, 8), (3, 7)])
def test_sharp_distributions(n, a, divergence):
    """Trained models are sharper than random init.  Own-action rows x 16 (twice the x 8 of _weights), moa_logits_w x 6 (MOA
    logits up to about +-7 on these inputs) and policy logits 6 randn (pi nearly one-hot for many agents); every 7th agent
    took an action of probability ~e^-30.  Every output is finite; the influence matches float64 from the kernel's own logits within
    OWN_TOL (1 + |v|); a JSD term is at most log 2.  pred and the counterfactual logits are compared with the oracle at 6 MOA_TOL:
    the error of h' (MOA_TOL, as the own-action rows enter in fp32 and the gate GEMM's operands are unchanged) reaches the logits
    through moa_logits_w, which is 6 times random init; h' and c' themselves at MOA_TOL."""
    from oracle import moa_ref
    policy = _policy()
    b = 300
    m = b * n
    w = policy.random_moa_weights(n, a, seed=60 + a)
    w["moa_lstm_w"][32:32 + a] *= 16.0
    w["moa_logits_w"] *= 6.0
    net = policy.MOANet(w, n)
    x, joint, _ = _inputs(b, n, a, seed=61, steps=1)[0]
    g = torch.Generator(device="cuda").manual_seed(62)
    pl = 6.0 * torch.randn((m, a), device="cuda", generator=g)
    rare = torch.arange(0, m, 7, device="cuda")
    own = joint.reshape(-1).long()
    pl[rare, own[rare]] = pl[rare].scatter(1, own[rare, None], -math.inf).max(dim=1).values - 30.0   # pi(own action) ~ e^-30
    hr = 0.5 * torch.randn((m, 128), device="cuda", generator=g)
    cr = 0.5 * torch.randn((m, 128), device="cuda", generator=g)
    h, c = net.state_from_rows(hr), net.state_from_rows(cr)
    s = net.step(x, joint, pl, h, c, divergence=divergence, counterfactuals=True)
    for name, t in (("pred", s.pred), ("influence", s.influence), ("influence_per_agent", s.influence_per_agent),
                    ("h", net.state_rows(s.h, m)), ("c", net.state_rows(s.c, m)), ("counterfactual", s.counterfactual)):
        assert bool(torch.isfinite(t).all()), name   # the state as agent rows: the tiled layout's padding rows are not written
    jn = _np(joint).astype(np.int64)
    ref = moa_ref.moa_forward(w, _np(x), jn, _np(pl), _np(hr), _np(cr), a, divergence=divergence)
    assert np.abs(ref["pred"]).max() > 5.0   # sharp: MOA logits of about +-7, softmax probabilities down to ~e^-14
    lp = torch.log_softmax(pl.double(), dim=1).gather(1, own[:, None])[:, 0]
    assert float(lp[rare].max()) < -29.0   # rare actions
    assert float((torch.softmax(pl.double(), dim=1).max(dim=1).values > 0.99).double().mean()) > 0.15   # near one-hot policies
    for name, got, tol in (("pred", s.pred, 6 * MOA_TOL), ("counterfactual", s.counterfactual, 6 * MOA_TOL),
                           ("h", net.state_rows(s.h, m), MOA_TOL), ("c", net.state_rows(s.c, m), MOA_TOL)):
        err = np.abs(_np(got) - ref[name]).max()
        assert err < tol, (name, err)
    ipa, infl = moa_ref.influence_from(_np(s.pred), _np(s.counterfactual), _np(pl), jn, a, divergence)
    for name, got, want in (("influence_per_agent", s.influence_per_agent, ipa), ("influence", s.influence, infl)):
        err = (np.abs(_np(got) - want) / (1 + np.abs(want))).max()
        assert err < OWN_TOL, (name, err)
    if divergence == "jsd":
        assert float(s.influence_per_agent.max()) <= math.log(2) + 1e-6
    assert infl.max() > 0.1   # not vacuous
    net.close()


def test_near_zero_influence():
    policy = _policy()
    n, a = 5, 8
    w = _weights(n, a, seed=11)
    w["moa_lstm_w"][32:32 + a] = 0.0   # the MOA ignores the own action
    net = policy.MOANet(w, n)
    x, joint, pl = _inputs(300, n, a, seed=12, steps=1)[0]
    h, c = net.initial_state(x.shape[0])
    assert float(net.step(x, joint, pl, h, c).influence.abs().max()) <= 1e-6
    net.close()
    net = policy.MOANet(_weights(n, a, seed=13), n)
    onehot = 100.0 * torch.nn.functional.one_hot(joint.reshape(-1).long(), a).float()   # pi one-hot at the action taken
    s = net.step(x, joint, onehot, h, c)
    assert float(s.influence.abs().max()) <= 1e-6
    assert float(net.step(x, joint, pl, h, c).influence.max()) > 1e-3   # not vacuous
    net.close()


def _rows_of(net, s, m):
    return [s.pred, s.influence, s.influence_per_agent, net.state_rows(s.h, m), net.state_rows(s.c, m)]


def test_per_agent_against_shared():
    policy = _policy()
    n, a, b = 5, 8, 300
    m = b * n
    w = _sets(n, a, n, seed=20)
    steps = _inputs(b, n, a, seed=21)
    shared, copies, per = policy.MOANet(w[0], n), policy.MOANet([w[0]] * n, n), policy.MOANet(w, n)
    singles = [policy.MOANet(ws, n) for ws in w]
    own = torch.arange(m, device="cuda") % n
    hs, cs = shared.initial_state(m)
    hp, cp = copies.initial_state(m)
    hq, cq = per.initial_state(m)
    hk = [net.initial_state(m) for net in singles]
    for x, joint, pl in steps:
        s1, s2, s3 = shared.step(x, joint, pl, hs, cs), copies.step(x, joint, pl, hp, cp), per.step(x, joint, pl, hq, cq)
        for got, want in zip(_rows_of(copies, s2, m), _rows_of(shared, s1, m)):
            assert torch.equal(got, want)
        sk = [net.step(x, joint, pl, *hc) for net, hc in zip(singles, hk)]
        for f, got in enumerate(_rows_of(per, s3, m)):
            want = torch.stack([_rows_of(singles[k], sk[k], m)[f] for k in range(n)])   # [n, m, ...]
            assert torch.equal(got, want[own, torch.arange(m, device="cuda")]), f
        hs, cs, hp, cp, hq, cq = s1.h, s1.c, s2.h, s2.c, s3.h, s3.c
        hk = [(s.h, s.c) for s in sk]
    for net in [shared, copies, per] + singles:
        net.close()


@pytest.mark.parametrize("kind,n,a", [pytest.param("shared", 5, 8, id="shared"), pytest.param("per_agent", 5, 8, id="per_agent"),
                                      pytest.param("shared", 16, 4, id="shared-16-4"), pytest.param("per_agent", 16, 4, id="per_agent-16-4"),
                                      pytest.param("shared", 5, 15, id="shared-5-15"), pytest.param("per_agent", 5, 15, id="per_agent-5-15")])
def test_scale_equals_one_group_per_cta_calls(kind, n, a):
    """At least four groups per CTA plus a ragged tail, against calls that each run at most one group per CTA."""
    policy = _policy()
    sms = _sms()
    per_policy = kind == "per_agent"
    ctas = sms // n if per_policy else sms
    rows = 4 * ctas * 128 + 77                     # agents per weight set
    b = rows if per_policy else -(-rows // n)
    m = b * n
    net = policy.MOANet(_sets(n, a, n if per_policy else 1, seed=30) if per_policy else _sets(n, a, 1, seed=30)[0], n)
    g = torch.Generator(device="cuda").manual_seed(31)
    h = net.state_from_rows(0.5 * torch.randn((m, 128), device="cuda", generator=g))
    c = net.state_from_rows(0.5 * torch.randn((m, 128), device="cuda", generator=g))
    x, joint, pl = _inputs(b, n, a, seed=32, steps=1)[0]
    big = net.step(x, joint, pl, h, c, counterfactuals=True)
    # chunks of whole envs and whole state groups: at most `ctas` groups per weight set
    env_chunk = ctas * 128 if per_policy else (ctas * 128 // (128 * n)) * 128
    parts = []
    hr, cr = net.state_rows(h, m), net.state_rows(c, m)
    for e0 in range(0, b, env_chunk):
        e1 = min(b, e0 + env_chunk)
        sl = slice(e0 * n, e1 * n)
        hh, cc = net.state_from_rows(hr[sl]), net.state_from_rows(cr[sl])
        s = net.step(x[sl], joint[e0:e1], pl[sl], hh, cc, counterfactuals=True)
        parts.append(_rows_of(net, s, (e1 - e0) * n) + [s.counterfactual])
    want = [torch.cat([p[f] for p in parts]) for f in range(6)]
    for f, got in enumerate(_rows_of(net, big, m) + [big.counterfactual]):
        assert torch.equal(got, want[f]), f
    assert len(parts) >= 4
    net.close()


def test_invalid_actions():
    """Envs 3, 7, 150 and 299 have one action -1, A, 127 or -128; the agent that took it has an invalid own action, whose extra
    drain (a' = A) runs on warps 0-3 for even A and on warps 4-7 for odd A: (N, A) = (5, 8), (5, 15) and (3, 7)."""
    for n, a in ((5, 8), (5, 15), (3, 7)):
        _check_invalid_actions(n, a)


def _check_invalid_actions(n, a):
    policy = _policy()
    b = 300
    m = b * n
    w = policy.random_moa_weights(n, a, seed=40)
    net = policy.MOANet(w, n)
    x, joint, pl = _inputs(b, n, a, seed=41, steps=1)[0]
    joint[3, 0], joint[7, 2 % n], joint[150, 4 % n], joint[299, 1] = -1, a, 127, -128
    bad = torch.zeros(b, dtype=torch.bool, device="cuda")
    bad[[3, 7, 150, 299]] = True
    bad = bad.repeat_interleave(n)
    h, c = net.initial_state(m)
    s = net.step(x, joint, pl, h, c, counterfactuals=True)
    assert bool(torch.isnan(s.influence[bad]).all()) and bool(torch.isnan(s.influence_per_agent[bad]).all()), (n, a)
    assert bool(torch.isfinite(s.influence[~bad]).all()) and bool(torch.isfinite(s.influence_per_agent[~bad]).all()), (n, a)
    ref = _oracle_rows([w], n, _np(x), _np(joint).astype(np.int64), _np(pl), np.zeros((m, 128)), np.zeros((m, 128)), a)
    for name, got in (("pred", s.pred), ("h", net.state_rows(s.h, m)), ("c", net.state_rows(s.c, m))):
        err = np.abs(_np(got) - ref[name]).max()
        assert err < MOA_TOL, (n, a, name, err)
    # wider integer dtypes are narrowed without wrapping: 136 is not action 8 - 128 + ...; -200 is not valid
    wide = joint.long()
    wide[3, 0], wide[7, 2] = 136, -200
    s2 = net.step(x, wide, pl, h, c)
    assert bool(torch.isnan(s2.influence[bad]).all()) and torch.equal(s2.influence[~bad], s.influence[~bad]), (n, a)
    net.close()


def test_closed_loop_harvest():
    """65 536 Harvest envs x 5 agents: policy_step -> MOANet.step -> env.step."""
    policy = _policy()
    from sequential_social_dilemma_games_b200.batched import BatchedSSDEnv, make_config
    n, b = 5, 65536
    m = b * n
    env = BatchedSSDEnv(make_config("harvest", num_agents=n), b, seed=3)
    pnet = policy.ConvToFCNet([policy.random_weights(num_outputs=8, seed=k) for k in range(n)])
    moa = policy.MOANet([policy.random_moa_weights(n, 8, seed=50 + k) for k in range(n)], n)
    pnet.seed_sampling(1)
    obs = env.reset()
    h, c = pnet.initial_state(m)
    hm, cm = moa.initial_state(m)
    for _ in range(4):
        x = pnet.features(obs)
        st = pnet.policy_step(obs, h, c)
        s = moa.step(x, st.actions.view(b, n), st.logits, hm, cm)
        for t in (s.pred, s.influence, s.influence_per_agent, s.h, s.c):
            assert bool(torch.isfinite(t).all())
        assert float(s.influence.min()) >= 0.0
        h, c, hm, cm = st.h, st.c, s.h, s.c
        obs, _ = env.step(st.actions.view(b, n))
    torch.cuda.synchronize()
    env.close()
    pnet.close()
    moa.close()


def test_errors():
    policy = _policy()
    from sequential_social_dilemma_games_b200 import _lib
    L = _lib.lib
    n, a, m = 5, 8, 20
    w = policy.random_moa_weights(n, a, seed=0)
    net = policy.MOANet(w, n)
    pnet = policy.ConvToFCNet(policy.random_weights(num_outputs=a, seed=0))
    p = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    x = torch.zeros((m, 32), device="cuda")
    joint = torch.zeros((m,), dtype=torch.int8, device="cuda")
    pl = torch.zeros((m, a), device="cuda")
    h, c = net.initial_state(m)
    hn, cn = torch.empty_like(h), torch.empty_like(c)
    pred, cf = torch.empty((m, n - 1, a), device="cuda"), torch.empty((m, a, n - 1, a), device="cuda")
    ipa, infl = torch.empty((m, n - 1), device="cuda"), torch.empty((m,), device="cuda")
    io = [p(x), p(joint), p(pl), p(h), p(c), p(hn), p(cn), p(pred), p(cf), p(ipa), p(infl)]
    step = lambda hd, *, mm=m, div=0, clip=math.inf, args=io: L.ssd_moa_step(hd, *args, mm, div, clip, st)
    assert step(net._h) == 0 and step(net._h, div=1) == 0 and step(net._h, mm=0) == 0
    assert L.ssd_moa_step(net._h, *io[:8], None, *io[9:], m, 0, math.inf, st) == 0   # counterfactual optional
    for k in range(11):
        if k == 8:
            continue
        args = list(io)
        args[k] = None
        assert step(net._h, args=args) == -1, k
    assert step(None) == -1
    assert step(net._h, mm=m - 1) == -1 and b"multiple" in L.ssd_last_error()
    assert step(net._h, mm=-5) == -1
    for div in (-1, 2, 7):
        assert step(net._h, div=div) == -1 and b"divergence" in L.ssd_last_error()
    for clip in (math.nan, -1.0):
        assert step(net._h, clip=clip) == -1 and b"clip" in L.ssd_last_error()
    args = list(io)
    args[0] = C.c_void_p(x.data_ptr() + 4)
    assert step(net._h, args=args) == -1 and b"aligned" in L.ssd_last_error()
    args = list(io)
    args[5], args[6] = args[3], args[4]
    assert step(net._h, args=args) == -1 and b"alias" in L.ssd_last_error()
    # handle crossing, both ways
    assert step(pnet._h) == -1 and b"MOA" in L.ssd_last_error()
    lg, vl = torch.zeros((m, a), device="cuda"), torch.zeros((m,), device="cuda")
    assert L.ssd_policy_lstm_heads(net._h, p(x), p(h), p(c), p(hn), p(cn), p(lg), p(vl), None, m, 0, 0, st) == -1
    assert b"MOA" in L.ssd_last_error()
    assert L.ssd_policy_lstm_heads_dist(net._h, p(x), p(h), p(c), p(hn), p(cn), p(lg), p(vl), 0, p(joint), None, None, m, 0, 0, st) == -1
    obs = torch.zeros((m, 15, 15, 3), dtype=torch.uint8, device="cuda")
    assert L.ssd_policy_features(net._h, p(obs), m, p(x), st) == -1 and b"MOA" in L.ssd_last_error()
    ids = torch.zeros((m,), dtype=torch.uint8, device="cuda")
    assert L.ssd_policy_pool_features(net._h, p(obs), p(ids), m, p(x), st) == -1
    z = np.zeros(4096, np.float32)
    zp = z.ctypes.data_as(C.c_void_p)
    assert L.ssd_policy_set_head_n(net._h, 1, 128, a, zp, zp, zp, zp, zp, zp, zp) == -1
    # creation: N, A, (N - 1) A, P, null pointers
    big = np.zeros((32 + 17 * 15) * 512 + 128 * 512 + 512 + 128 * 64 * 16 + 64 * 16, np.float32)
    bp = big.ctypes.data_as(C.c_void_p)
    out = C.c_void_p()
    for nn, aa, pp in ((1, 8, 1), (17, 2, 1), (5, 0, 1), (5, 16, 1), (9, 9, 1), (5, 8, 2), (5, 8, 0), (5, 8, 4)):
        assert L.ssd_moa_create(0, pp, nn, aa, bp, bp, bp, bp, bp, C.byref(out)) == -1, (nn, aa, pp)
        assert not out.value
    assert L.ssd_moa_create(0, 1, 5, 8, bp, None, bp, bp, bp, C.byref(out)) == -1
    assert L.ssd_moa_create(0, 1, 5, 8, bp, bp, bp, bp, bp, None) == -1
    assert L.ssd_moa_create(0, 1, 9, 8, bp, bp, bp, bp, bp, C.byref(out)) == 0   # (N - 1) A = 64
    L.ssd_moa_destroy(out)
    torch.cuda.synchronize()
    # Python
    for kw in ({"divergence": "KL"}, {"divergence": None}, {"clip": float("nan")}, {"clip": -1.0}):
        with pytest.raises(ValueError):
            net.step(x, joint, pl, h, c, **kw)
    for bad in (joint[:5], joint.float(), joint.cpu(), joint.tolist()):
        with pytest.raises(ValueError):
            net.step(x, bad, pl, h, c)
    for bad in (pl[:, :5], pl.double(), pl.cpu()):
        with pytest.raises(ValueError):
            net.step(x, joint, bad, h, c)
    with pytest.raises(ValueError):
        net.step(x[:7], joint[:7], pl[:7], h, c)
    with pytest.raises(ValueError):
        net.step(x.double(), joint, pl, h, c)
    with pytest.raises(ValueError):
        policy.MOANet([w, w], n)
    with pytest.raises(ValueError):
        policy.MOANet(w, 4)
    net.close()
    pnet.close()
