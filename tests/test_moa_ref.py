"""The float64 restatement of the model of other agents and the influence reward (oracle/moa_ref.py), checked without a GPU: a
hand-computed vector, the two cases where the influence must vanish, the Jensen-Shannon bound and the order of the one-hot
input rows."""
import math

import numpy as np

from oracle import moa_ref


def _weights(n, a, u, seed):
    rng = np.random.RandomState(seed)
    return {"moa_lstm_w": 0.3 * rng.randn(32 + n * a, 4 * u), "moa_lstm_u": 0.3 * rng.randn(u, 4 * u), "moa_lstm_b": 0.1 * rng.randn(4 * u),
            "moa_logits_w": rng.randn(u, (n - 1) * a), "moa_logits_b": 0.1 * rng.randn((n - 1) * a)}


def _case(n, a, b, seed, u=16):
    rng = np.random.RandomState(seed + 1)
    m = b * n
    return (_weights(n, a, u, seed), rng.randn(m, 32), rng.randint(0, a, size=(b, n)), 2 * rng.randn(m, a), 0.5 * rng.randn(m, u),
            0.5 * rng.randn(m, u))


def test_hand_vector_two_agents_two_actions():
    """N = 2, A = 2, one LSTM unit, x = h = c = 0: the gates are the sum of the own row and the other's row."""
    w = {"moa_lstm_w": np.zeros((36, 4)), "moa_lstm_u": np.zeros((1, 4)), "moa_lstm_b": np.zeros(4),
         "moa_logits_w": np.array([[1.0, -1.0]]), "moa_logits_b": np.array([0.5, 0.0])}
    w["moa_lstm_w"][32] = [1.0, 0.0, 2.0, 0.0]    # own action 0: i, f, c~, o
    w["moa_lstm_w"][33] = [0.0, 0.0, -1.0, 1.0]   # own action 1
    w["moa_lstm_w"][34] = [0.0, 0.0, 0.0, 0.5]    # the other agent's action 0
    w["moa_lstm_w"][35] = [0.5, 0.0, 0.0, 0.0]    # the other agent's action 1
    joint = np.array([[0, 1]])                    # agent 0 took 0, agent 1 took 1
    pl = np.array([[0.0, math.log(3.0)], [0.0, 0.0]])   # pi_0 = (1/4, 3/4), pi_1 = (1/2, 1/2)
    sig = lambda z: 1.0 / (1.0 + math.exp(-z))

    def logits(zi, zc, zo):
        cc = sig(zi) * math.tanh(zc)
        hh = sig(zo) * math.tanh(cc)
        return np.array([hh + 0.5, -hh]), hh, cc

    # agent 0 (own 0, other 1): own row 32 or 33, other row 35
    l00, h0, c0 = logits(1.0 + 0.5, 2.0, 0.0)
    l01, _, _ = logits(0.0 + 0.5, -1.0, 1.0)
    # agent 1 (own 1, other 0): own row 32 or 33, other row 34
    l10, _, _ = logits(1.0, 2.0, 0.5)
    l11, h1, c1 = logits(0.0, -1.0, 1.5)
    out = moa_ref.moa_forward(w, np.zeros((2, 32)), joint, pl, np.zeros((2, 1)), np.zeros((2, 1)), 2)
    np.testing.assert_allclose(out["pred"][:, 0], [l00, l11], rtol=0, atol=1e-15)
    np.testing.assert_allclose(out["h"][:, 0], [h0, h1], atol=1e-15)
    np.testing.assert_allclose(out["c"][:, 0], [c0, c1], atol=1e-15)
    np.testing.assert_allclose(out["counterfactual"][0, :, 0], [l00, l01], atol=1e-15)
    np.testing.assert_allclose(out["counterfactual"][1, :, 0], [l10, l11], atol=1e-15)
    sm = lambda l: np.exp(l) / np.exp(l).sum()
    for m, (pi, cfs, act) in enumerate((((0.25, 0.75), (l00, l01), 0), ((0.5, 0.5), (l10, l11), 1))):
        q = pi[0] * sm(cfs[0]) + pi[1] * sm(cfs[1])
        p = sm(cfs[act])
        kl = float((p * np.log(p / q)).sum())
        mu = 0.5 * (p + q)
        jsd = float(0.5 * (p * np.log(p / mu)).sum() + 0.5 * (q * np.log(q / mu)).sum())
        assert abs(out["influence_per_agent"][m, 0] - kl) < 1e-15 and abs(out["influence"][m] - kl) < 1e-15
        ipa, _ = moa_ref.influence_from(out["pred"], out["counterfactual"], pl, joint, 2, "jsd")
        assert abs(ipa[m, 0] - jsd) < 1e-15
        assert kl > 1e-3


def test_no_influence_without_own_action_rows():
    w, x, joint, pl, h, c = _case(5, 8, 7, seed=1)
    w["moa_lstm_w"][32:40] = 0.0
    out = moa_ref.moa_forward(w, x, joint, pl, h, c, 8)
    assert np.abs(out["influence"]).max() < 1e-12 and np.abs(out["influence_per_agent"]).max() < 1e-12
    assert np.abs(out["pred"]).max() > 0.1


def test_no_influence_with_a_deterministic_policy():
    w, x, joint, pl, h, c = _case(5, 9, 7, seed=2)
    pl = np.where(np.arange(9)[None, :] == joint.reshape(-1, 1), 100.0, 0.0)   # pi one-hot at the action taken
    out = moa_ref.moa_forward(w, x, joint, pl, h, c, 9)
    assert np.abs(out["influence"]).max() < 1e-12
    pl_rand = np.random.RandomState(3).randn(*pl.shape)
    assert moa_ref.moa_forward(w, x, joint, pl_rand, h, c, 9)["influence"].min() > 1e-6   # not vacuous


def test_jsd_is_bounded_by_log_two_and_the_clip_clamps():
    w, x, joint, pl, h, c = _case(3, 4, 20, seed=4)
    w["moa_logits_w"] *= 30.0   # sharp predictions: divergences near their bound
    jsd = moa_ref.moa_forward(w, x, joint, pl, h, c, 4, divergence="jsd")
    assert (jsd["influence_per_agent"] >= -1e-15).all() and (jsd["influence_per_agent"] <= math.log(2) + 1e-15).all()
    assert jsd["influence_per_agent"].max() > 0.3
    kl = moa_ref.moa_forward(w, x, joint, pl, h, c, 4, clip=0.25)
    assert kl["influence"].max() <= 0.25 and (kl["influence"] == 0.25).any()


def test_own_and_other_rows_follow_agent_order():
    """Exchanging the actions of agents 1 and 2 equals exchanging their one-hot row blocks and logit columns, for agent 0."""
    n, a = 3, 4
    w, x, joint, pl, h, c = _case(n, a, 11, seed=5)
    swapped = joint[:, [0, 2, 1]]
    w2 = {k: v.copy() for k, v in w.items()}
    blk = lambda s: slice(32 + a + s * a, 32 + a + (s + 1) * a)
    w2["moa_lstm_w"][blk(0)], w2["moa_lstm_w"][blk(1)] = w["moa_lstm_w"][blk(1)], w["moa_lstm_w"][blk(0)]
    col = np.r_[a:2 * a, 0:a]
    w2["moa_logits_w"], w2["moa_logits_b"] = w["moa_logits_w"][:, col], w["moa_logits_b"][col]
    ref = moa_ref.moa_forward(w, x, joint, pl, h, c, a)
    got = moa_ref.moa_forward(w2, x, swapped, pl, h, c, a)
    agent0 = np.arange(0, x.shape[0], n)
    np.testing.assert_allclose(got["pred"][agent0][:, [1, 0]], ref["pred"][agent0], atol=1e-12)
    np.testing.assert_allclose(got["h"][agent0], ref["h"][agent0], atol=1e-12)
    np.testing.assert_allclose(got["influence_per_agent"][agent0][:, [1, 0]], ref["influence_per_agent"][agent0], atol=1e-12)
    # the own slot comes first: agent 1's own action is row block 0 (rows 32 .. 32 + A)
    w3 = {k: v.copy() for k, v in w.items()}
    w3["moa_lstm_w"][32:32 + a] += 1.0
    moved = moa_ref.moa_forward(w3, x, joint, pl, h, c, a)
    assert np.abs(moved["pred"] - ref["pred"]).min() > 0


def test_invalid_actions_poison_their_env_only():
    w, x, joint, pl, h, c = _case(4, 5, 6, seed=6)
    joint[2, 1], joint[4, 3] = -1, 5
    out = moa_ref.moa_forward(w, x, joint, pl, h, c, 5)
    bad = np.zeros(6, bool)
    bad[[2, 4]] = True
    bad = np.repeat(bad, 4)
    assert np.isnan(out["influence"][bad]).all() and np.isnan(out["influence_per_agent"][bad]).all()
    assert np.isfinite(out["influence"][~bad]).all() and np.isfinite(out["pred"]).all()
