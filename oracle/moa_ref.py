"""TEST INFRASTRUCTURE ONLY (see oracle/README.md): float64 numpy restatement of the model of other agents (MOA) and the
social-influence reward of the reference's causal-influence models (models/moa_model.py MOA_LSTM, common_funcs.py
compute_influence_reward; SURVEY.md rows 11 and 12), the checker of csrc/ssd_policy_moa.cu.  The repository has no copy of
those files, so this is the library's contract as include/ssd_b200.h states it (the structure of Jaques et al. 2019):

  agent m = b * N + i, input(a') = [x | onehot(a') | onehot(a_{b,j}) for j != i in increasing j]   (an invalid action: zeros)
  LSTM(128) as policy_ref.lstm_step on the weights moa_lstm_w / moa_lstm_u / moa_lstm_b, then Dense((N-1) * A)
  pred = the logits at the actual joint action; counterfactual[m, a'] = the logits with the own slot set to onehot(a')
  q_k = sum_a' softmax(policy_logits)[a'] softmax(counterfactual[m, a', k]), renormalised to sum 1
  influence_per_agent[m, k] = KL(softmax(pred[m, k]) || q_k) (terms with p = 0 skipped) or the Jensen-Shannon divergence
  influence[m] = clamp(sum_k influence_per_agent[m, k], -clip, clip); NaN for every agent of an env with an invalid action."""
import numpy as np

from .policy_ref import lstm_step


def _lstm_weights(w):
    return {"lstm_w": w["moa_lstm_w"], "lstm_u": w["moa_lstm_u"], "lstm_b": w["moa_lstm_b"]}


def moa_input(x, joint, num_actions, own=None):
    """[M, 32 + N A] inputs of agents m = b * N + i; joint int [B, N]; `own` [M] replaces the own slot's action if given."""
    joint = np.asarray(joint).astype(np.int64)
    b_count, n = joint.shape
    a_count = num_actions
    m = b_count * n
    onehot = lambda a: np.where(((a >= 0) & (a < a_count))[:, None], np.eye(a_count)[np.clip(a, 0, a_count - 1)], 0.0)
    own_a = joint.reshape(-1) if own is None else np.asarray(own).astype(np.int64)
    cols = [np.asarray(x, np.float64), onehot(own_a)]
    idx = np.arange(m)
    b, i = idx // n, idx % n
    for k in range(n - 1):
        j = np.where(k < i, k, k + 1)
        cols.append(onehot(joint[b, j]))
    return np.concatenate(cols, axis=1)


def moa_step(w, x, joint, h, c, num_actions, own=None):
    """-> (logits [M, N-1, A], h', c') of one MOA step."""
    n = np.asarray(joint).shape[1]
    h2, c2 = lstm_step(_lstm_weights(w), moa_input(x, joint, num_actions, own), np.asarray(h, np.float64), np.asarray(c, np.float64))
    y = h2 @ w["moa_logits_w"].astype(np.float64) + w["moa_logits_b"].astype(np.float64)
    return y.reshape(-1, n - 1, num_actions), h2, c2


def counterfactuals(w, x, joint, h, c, num_actions):
    """[M, A, N-1, A]: the logits with every agent's own action set to a', from the same (h, c)."""
    m = np.asarray(x).shape[0]
    return np.stack([moa_step(w, x, joint, h, c, num_actions, own=np.full(m, a))[0] for a in range(num_actions)], axis=1)


def _softmax(z, axis=-1):
    z = np.asarray(z, np.float64)
    e = np.exp(z - z.max(axis=axis, keepdims=True))
    return e / e.sum(axis=axis, keepdims=True)


def _kl(p, q):
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(p > 0, p * (np.log(p) - np.log(q)), 0.0).sum(axis=-1)


def influence_from(pred, cf, policy_logits, joint, num_actions, divergence="kl", clip=np.inf):
    """(influence_per_agent [M, N-1], influence [M]) from the logits: pred [M, N-1, A], cf [M, A, N-1, A]."""
    pi = _softmax(policy_logits)                                          # [M, A]
    q = np.einsum("ma,makx->mkx", pi, _softmax(cf))                       # [M, N-1, A]
    q = q / q.sum(axis=-1, keepdims=True)
    p = _softmax(pred)
    if divergence == "kl":
        d = _kl(p, q)
    elif divergence == "jsd":
        mu = 0.5 * (p + q)
        d = 0.5 * _kl(p, mu) + 0.5 * _kl(q, mu)
    else:
        raise ValueError(divergence)
    joint = np.asarray(joint).astype(np.int64)
    bad = np.repeat(((joint < 0) | (joint >= num_actions)).any(axis=1), joint.shape[1])
    d[bad] = np.nan
    return d, np.clip(d.sum(axis=1), -clip, clip)


def moa_forward(w, x, joint, policy_logits, h, c, num_actions, divergence="kl", clip=np.inf):
    """-> dict pred, h, c, counterfactual, influence_per_agent, influence (all float64)."""
    pred, h2, c2 = moa_step(w, x, joint, h, c, num_actions)
    cf = counterfactuals(w, x, joint, h, c, num_actions)
    ipa, infl = influence_from(pred, cf, policy_logits, joint, num_actions, divergence, clip)
    return {"pred": pred, "h": h2, "c": c2, "counterfactual": cf, "influence_per_agent": ipa, "influence": infl}
