"""One network per agent id (ConvToFCNet([weights_0, ..., weights_{P-1}]), ssd_policy_create_n / ssd_policy_set_head_n): agent
(b, p) of a [B, P, 15, 15, 3] batch is evaluated with weights_p by the per-agent variants of the two fused kernels.  Each agent
runs the same instruction sequence on the same weights as in the shared network, so the comparisons with the shared network
and with P separate networks are bitwise; the float64 oracle (oracle/policy_ref.py) bounds each column to the tolerances of
test_policy_gpu.py."""
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


@pytest.fixture(scope="module")
def env_obs():
    """Three consecutive observation tensors of 3 200 Harvest envs x 5 agents from the step kernel, flattened to 16 000 agents."""
    from sequential_social_dilemma_games_b200.batched import BatchedSSDEnv, make_config
    env = BatchedSSDEnv(make_config("harvest", num_agents=5), 3200, seed=9)
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(4)
    out = []
    for _ in range(3):
        a = torch.randint(0, NUM_OUTPUTS, (3200, 5), dtype=torch.int8, device="cuda", generator=g)
        obs, _ = env.step(a)
        out.append(obs.reshape(-1, 15, 15, 3).clone())
    torch.cuda.synchronize()
    env.close()
    return out


def _obs_steps(source, B, P, env_obs, seed):
    if source == "env":   # the first B * P agents of the step kernel's output, regrouped as [B, P]
        return [o[:B * P].reshape(B, P, 15, 15, 3) for o in env_obs]
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randint(0, 256, (B, P, 15, 15, 3), dtype=torch.uint8, device="cuda", generator=g) for _ in range(3)]


@pytest.mark.parametrize("source", ["random", "env"])
@pytest.mark.parametrize("P", [2, 5, 16])
@pytest.mark.parametrize("B", [1, 127, 128, 129, 1000])
def test_identical_weights_reproduce_shared_net(B, P, source, env_obs):
    """P copies of one weight set == the shared network, bitwise: features, logits, value, h and c over three recurrent
    steps, and the sampled actions for the same (seed, counter)."""
    policy = _policy()
    w = policy.random_weights(num_outputs=NUM_OUTPUTS, seed=21)
    shared, per = policy.ConvToFCNet(w), policy.ConvToFCNet([w] * P)
    assert per.num_policies == P
    M = B * P
    steps = _obs_steps(source, B, P, env_obs, seed=B * 100 + P)
    assert torch.equal(per.features(steps[0]), shared.features(steps[0].reshape(M, 15, 15, 3)))
    assert torch.equal(per.features(steps[0].reshape(M, 15, 15, 3)), shared.features(steps[0]))
    hs, cs = shared.initial_state(M)
    hp, cp = per.initial_state(M)
    assert hp.shape == (P * ((B + 127) // 128), 8, 128, 16)
    shared.seed_sampling(1234)
    per.seed_sampling(1234)
    for obs in steps:
        ls, vs, hs2, cs2 = shared.forward(obs, hs, cs)
        lp, vp, hp2, cp2 = per.forward(obs, hp, cp)
        assert torch.equal(lp, ls) and torch.equal(vp, vs)
        assert torch.equal(per.state_rows(hp2, M), shared.state_rows(hs2, M))
        assert torch.equal(per.state_rows(cp2, M), shared.state_rows(cs2, M))
        a_s, v_s, hs, cs = shared.act(obs, hs, cs)
        a_p, v_p, hp, cp = per.act(obs, hp, cp)
        assert torch.equal(a_p, a_s) and torch.equal(v_p, v_s)
        assert torch.equal(per.state_rows(hp, M), shared.state_rows(hs, M))
    assert ls.abs().max().item() > 0.01   # not all zero
    shared.close()
    per.close()


def test_state_rows_round_trip():
    policy = _policy()
    per = policy.ConvToFCNet([policy.random_weights(num_outputs=NUM_OUTPUTS, seed=s) for s in range(5)])
    for m in (5, 5 * 129, 5 * 1000):
        rows = torch.arange(m * 128.0, device="cuda").reshape(m, 128)
        tiled = per.state_from_rows(rows)
        assert tiled.shape == (5 * ((m // 5 + 127) // 128), 8, 128, 16)
        assert torch.equal(per.state_rows(tiled, m), rows)
        g = tiled.shape[0] // 5   # element (agent b * P + p, unit u) in state group p * G + b / 128
        b, p, u = m // 5 - 1, 3, 37
        assert tiled[p * g + b // 128, u // 16, b % 128, u % 16].item() == rows[b * 5 + p, u].item()
    per.close()


def _distinct(P=5, num_outputs=NUM_OUTPUTS):
    policy = _policy()
    return [policy.random_weights(num_outputs=num_outputs, seed=100 + p) for p in range(P)]


@pytest.mark.parametrize("B,num_outputs", [pytest.param(B, NUM_OUTPUTS, id=str(B)) for B in (1, 129, 1000)]
                         + [pytest.param(B, A, id="%d-outputs%d" % (B, A)) for A in (1, 15) for B in (1, 129, 1000)])
def test_distinct_weights_match_separate_nets(B, num_outputs):
    """Column p of a P = 5 network == ConvToFCNet(weights[p]) on obs[:, p], bitwise (features, three recurrent steps), and
    within the kernels' tolerances of the float64 oracle with weights[p].  1 and 15 outputs put the value in head column 1 and
    15, which the per-agent head selects with code of its own."""
    from oracle import policy_ref
    policy = _policy()
    P, M = 5, B * 5
    ws = _distinct(P, num_outputs)
    per = policy.ConvToFCNet(ws)
    singles = [policy.ConvToFCNet(w) for w in ws]
    steps = _obs_steps("random", B, P, None, seed=B)
    feats = per.features(steps[0]).reshape(B, P, 32)
    for p in range(P):
        col = steps[0][:, p].clone()   # a copy: for B = 1 the view is contiguous but not 16-byte aligned
        assert torch.equal(feats[:, p], singles[p].features(col))
        err = np.abs(feats[:, p].cpu().numpy().astype(np.float64) - policy_ref.features(ws[p], col.cpu().numpy())).max()
        assert err < TRUNK_TOL, (p, err)
    hp, cp = per.initial_state(M)
    hs = [s.initial_state(B) for s in singles]
    h64 = [(np.zeros((B, 128)), np.zeros((B, 128))) for _ in range(P)]
    for obs in steps:
        logits, value, hp2, cp2 = per.forward(obs, hp, cp)
        hp, cp = hp2, cp2
        rows_h, rows_c = per.state_rows(hp2, M).reshape(B, P, 128), per.state_rows(cp2, M).reshape(B, P, 128)
        logits, value = logits.reshape(B, P, num_outputs), value.reshape(B, P)
        for p in range(P):
            col = obs[:, p].clone()
            l1, v1, h1, c1 = singles[p].forward(col, *hs[p])
            hs[p] = (h1, c1)
            assert torch.equal(logits[:, p], l1) and torch.equal(value[:, p], v1)
            assert torch.equal(rows_h[:, p], singles[p].state_rows(h1, B)) and torch.equal(rows_c[:, p], singles[p].state_rows(c1, B))
            l64, v64, hh, cc = policy_ref.forward(ws[p], col.cpu().numpy(), *h64[p])
            h64[p] = (hh, cc)
            for got, want in ((logits[:, p], l64), (value[:, p], v64), (rows_h[:, p], hh), (rows_c[:, p], cc)):
                assert np.abs(got.cpu().numpy().astype(np.float64) - want).max() < FWD_TOL
    per.close()
    for s in singles:
        s.close()


def test_distinct_weights_actions_follow_agent_major_index():
    """Over three recurrent steps, the sampled actions of column p == those of ConvToFCNet(weights[p]) run on a batch with
    column p's observations in every column, at column p, for the same (seed, counter): both key Philox by the agent-major
    index b * P + p and see the same logits there.  (ConvToFCNet(weights[p]) on obs[:, p] alone numbers its agents b.)"""
    policy = _policy()
    B, P = 1000, 5
    ws = _distinct(P)
    per = policy.ConvToFCNet(ws)
    steps = _obs_steps("random", B, P, None, seed=8)
    per.seed_sampling(5)
    h, c = per.initial_state(B * P)
    acts = []
    for obs in steps:
        a, _, h, c = per.act(obs, h, c)
        acts.append(a.reshape(B, P))
    for p in range(P):
        single = policy.ConvToFCNet(ws[p])
        single.seed_sampling(5)
        h1, c1 = single.initial_state(B * P)
        for k, obs in enumerate(steps):
            same = obs[:, p:p + 1].expand(B, P, 15, 15, 3).contiguous()
            a1, _, h1, c1 = single.act(same, h1, c1)
            assert torch.equal(acts[k][:, p], a1.reshape(B, P)[:, p]), (p, k)
        single.close()
    assert len(torch.unique(torch.stack(acts))) > 1
    assert not torch.equal(acts[0], acts[1])   # a fresh counter every step
    per.close()


def test_weight_order_is_column_order():
    """Reversing the weight list (and the columns) reverses the outputs, bitwise; different policies differ by far more than
    the kernels' tolerance."""
    policy = _policy()
    B, P = 300, 5
    ws = _distinct(P)
    for w in ws:   # spread the logits of the random init so that policies differ there by far more than FWD_TOL as well
        w["logits_w"] = (w["logits_w"] * 16).astype(np.float32)
    fwd, rev = policy.ConvToFCNet(ws), policy.ConvToFCNet(ws[::-1])
    obs = torch.randint(0, 256, (B, P, 15, 15, 3), dtype=torch.uint8, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    obs_rev = obs.flip(1).contiguous()
    M = B * P
    l1, v1, h1, c1 = fwd.forward(obs, *fwd.initial_state(M))
    l2, v2, h2, c2 = rev.forward(obs_rev, *rev.initial_state(M))
    assert torch.equal(fwd.features(obs).reshape(B, P, 32), rev.features(obs_rev).reshape(B, P, 32).flip(1))
    assert torch.equal(l1.reshape(B, P, -1), l2.reshape(B, P, -1).flip(1))
    assert torch.equal(v1.reshape(B, P), v2.reshape(B, P).flip(1))
    assert torch.equal(fwd.state_rows(h1, M).reshape(B, P, -1), rev.state_rows(h2, M).reshape(B, P, -1).flip(1))
    assert torch.equal(fwd.state_rows(c1, M).reshape(B, P, -1), rev.state_rows(c2, M).reshape(B, P, -1).flip(1))
    # the same observation in every column: the columns differ only by their weights
    same = obs[:, :1].expand(B, P, 15, 15, 3).contiguous()
    f = fwd.features(same).reshape(B, P, 32)
    lg = fwd.forward(same, *fwd.initial_state(M))[0].reshape(B, P, -1)
    for p in range(1, P):
        assert (f[:, p] - f[:, 0]).abs().max().item() > 100 * TRUNK_TOL, p
        assert (lg[:, p] - lg[:, 0]).abs().max().item() > 20 * FWD_TOL, p
    fwd.close()
    rev.close()


def test_closed_loop_per_agent_policies():
    """BatchedSSDEnv (300 Harvest envs x 5 agents) -> per-agent act -> env for six steps, all on the device; the same seeds
    give the same actions."""
    policy = _policy()
    from sequential_social_dilemma_games_b200.batched import BatchedSSDEnv, make_config
    ws = _distinct(5)

    def run():
        env = BatchedSSDEnv(make_config("harvest", num_agents=5), 300, seed=5)
        net = policy.ConvToFCNet(ws)
        net.seed_sampling(42)
        obs = env.reset()
        h, c = net.initial_state(300 * 5)
        acts = []
        for _ in range(6):
            a, value, h, c = net.act(obs, h, c)          # obs [300, 5, 15, 15, 3] straight from the step kernel
            acts.append(a)
            obs, rew = env.step(a.view(300, 5))
        torch.cuda.synchronize()
        env.close()
        net.close()
        return torch.stack(acts)

    a1, a2 = run(), run()
    assert a1.dtype == torch.int8 and int(a1.min()) >= 0 and int(a1.max()) < NUM_OUTPUTS
    assert torch.equal(a1, a2)
    assert len(torch.unique(a1)) > 1


def test_errors():
    policy = _policy()
    from sequential_social_dilemma_games_b200 import _lib
    L = _lib.lib
    w = policy.random_weights(num_outputs=NUM_OUTPUTS, seed=0)
    per = policy.ConvToFCNet([w, w])
    # M % P != 0, wrong column count, other entry points
    with pytest.raises(ValueError):
        per.features(torch.zeros((7, 15, 15, 3), dtype=torch.uint8, device="cuda"))
    with pytest.raises(ValueError):
        per.features(torch.zeros((4, 3, 15, 15, 3), dtype=torch.uint8, device="cuda"))
    with pytest.raises(ValueError):
        per.initial_state(7)
    with pytest.raises(ValueError):
        per.forward_unfused(torch.zeros((4, 2, 15, 15, 3), dtype=torch.uint8, device="cuda"), *per.initial_state(8))
    obs = torch.zeros((8, 15, 15, 3), dtype=torch.uint8, device="cuda")
    feats = torch.zeros((8, 32), device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: C.c_void_p(t.data_ptr())
    assert L.ssd_policy_features(per._h, p(obs), 7, p(feats), st) == -1 and b"multiple" in L.ssd_last_error()
    h, c = per.initial_state(8)
    lg, vl = torch.zeros((8, NUM_OUTPUTS), device="cuda"), torch.zeros((8,), device="cuda")
    assert L.ssd_policy_lstm_heads(per._h, p(feats), p(h), p(c), p(h), p(c), p(lg), p(vl), None, 7, 0, 0, st) == -1
    assert b"multiple" in L.ssd_last_error()
    # P = 0, P > 16
    with pytest.raises(ValueError):
        policy.ConvToFCNet([])
    with pytest.raises(_lib.SsdError):
        policy.ConvToFCNet([w] * 17)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    tw = [np.ascontiguousarray(w[k]) for k in ("conv_w", "conv_b", "fc1_w", "fc1_b", "fc2_w", "fc2_b")]
    hw = [np.ascontiguousarray(w[k]) for k in ("lstm_w", "lstm_u", "lstm_b", "logits_w", "logits_b", "value_w", "value_b")]
    hh = C.c_void_p()
    for bad in (0, 17, -1):
        assert L.ssd_policy_create_n(7, 0, bad, *[ptr(a) for a in tw], C.byref(hh)) == -1 and not hh.value
    # a head P that differs from the trunk P (and the P = 1 entry point on a P = 2 handle)
    assert L.ssd_policy_set_head_n(per._h, 3, 128, NUM_OUTPUTS, *[ptr(a) for a in hw]) == -1 and b"trunk" in L.ssd_last_error()
    assert L.ssd_policy_set_head(per._h, 128, NUM_OUTPUTS, *[ptr(a) for a in hw]) == -1
    assert L.ssd_policy_set_head_n(per._h, 0, 128, NUM_OUTPUTS, *[ptr(a) for a in hw]) == -1
    # mismatched weight shapes; a cell that the fused head does not take
    w9 = policy.random_weights(num_outputs=9, seed=1)
    with pytest.raises(ValueError):
        policy.ConvToFCNet([w, w9])
    w_trunk = dict(w)
    w_trunk["fc1_w"] = np.zeros((1000, 32), np.float32)
    with pytest.raises(ValueError):
        policy.ConvToFCNet([w, w_trunk])
    with pytest.raises(ValueError):
        policy.ConvToFCNet([policy.random_weights(num_outputs=NUM_OUTPUTS, cell_size=64, seed=s) for s in range(2)])
    with pytest.raises(ValueError):
        policy.ConvToFCNet([{k: v for k, v in w.items() if not k.startswith(("lstm", "logits", "value"))}] * 2)
    # P = 1 given as a list is the shared network, unfused route included
    one = policy.ConvToFCNet([policy.random_weights(num_outputs=NUM_OUTPUTS, cell_size=64, seed=2)])
    assert one.num_policies == 1 and not one._fused_head
    one.close()
    per.close()

