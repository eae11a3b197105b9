"""TEST INFRASTRUCTURE ONLY (see oracle/README.md): float64 restatement of the advantages and value targets the rollout worker
computes for the reference's trainers (algorithms/{ppo,a3c,impala}_causal.py), the checker of csrc/ssd_advantages.cu.  The
reference's checkout and ray are not part of this repository, so this is the library's contract as include/ssd_b200.h states it,
written the way RLlib (ray 0.7.6) writes it and deliberately not in the kernel's algebra:

  inputs [T, M] (agent m of env b = m // N), dones [T, B]; the step reward r_t = rewards_t + w * intrinsic_t;
  every column is split into episode fragments at the dones: a fragment ends with a done step or with step T-1, and its last_r
  is 0 after a done and bootstrap[m] otherwise (RLlib runs every fragment separately);
  compute_advantages(use_gae=True):  vpred = [V, last_r]; delta_t = r_t + gamma vpred_{t+1} - vpred_t;
                                     advantages = discount(delta, gamma lambda); value_targets = advantages + V
  compute_advantages(use_gae=False): advantages = discount([r, last_r], gamma)[:-1]  (no value targets)
  vtrace.from_importance_weights:    rho = exp(target_logp - behaviour_logp), rho_bar = min(clip_rho, rho), c = min(1, rho),
                                     rho_pg = min(clip_pg_rho, rho) (a threshold of +inf: no clip, None in RLlib);
                                     V_{t+1} = [V[1:], last_r]; delta_t = rho_bar_t (r_t + gamma V_{t+1} - V_t);
                                     acc = 0; for t backwards: acc = delta_t + gamma c_t acc; vs_t = acc + V_t;
                                     vs_{t+1} = [vs[1:], last_r]; pg_advantages = rho_pg_t (r_t + gamma vs_{t+1} - V_t)
  with discount(x, g) = scipy.signal.lfilter([1], [1, -g], x[::-1])[::-1], RLlib's discount.

`error_bound` is the fp32 bound the GPU tests hold the kernel to (DESIGN.md section 5.8)."""
import numpy as np
import scipy.signal

U = 2.0 ** -24   # unit roundoff of fp32


def discount(x, gamma):
    return scipy.signal.lfilter([1], [1, -float(gamma)], np.asarray(x, np.float64)[::-1], axis=0)[::-1]


def _columns(rewards, values, dones, intrinsic, w):
    """-> rewards + w * intrinsic and values as float64 [T, M], and the dones of every column as bool [T, M]."""
    values = np.asarray(values, np.float64)
    t_count, m = values.shape
    dones = np.asarray(dones).reshape(t_count, -1) != 0
    n = m // dones.shape[1]
    assert n * dones.shape[1] == m, "M must be a multiple of B"
    r = np.asarray(rewards).astype(np.float64)
    if intrinsic is not None:
        r = r + float(w) * np.asarray(intrinsic, np.float64)
    return r, values, np.repeat(dones, n, axis=1)


def fragments(done_col, bootstrap):
    """[(start, end, last_r)] of one column: end exclusive; last_r 0 after a done, the bootstrap after step T-1."""
    out, start = [], 0
    for t in np.flatnonzero(done_col):
        out.append((start, t + 1, 0.0))
        start = t + 1
    if start < len(done_col):
        out.append((start, len(done_col), float(bootstrap)))
    return out


def compute_advantages_fragment(rewards, vf_preds, last_r, gamma, lambda_, use_gae):
    """RLlib's compute_advantages on one fragment -> (advantages, value_targets or None)."""
    if use_gae:
        vpred_t = np.concatenate([vf_preds, [last_r]])
        delta_t = rewards + gamma * vpred_t[1:] - vpred_t[:-1]
        adv = discount(delta_t, gamma * lambda_)
        return adv, adv + vf_preds
    return discount(np.concatenate([rewards, [last_r]]), gamma)[:-1], None


def compute_advantages(rewards, values, dones, bootstrap, gamma, lambda_, use_gae=True, intrinsic=None, intrinsic_weight=0.0):
    """[T, M] float64 advantages and value targets (None for use_gae=False) of every column, fragment by fragment."""
    r, v, d = _columns(rewards, values, dones, intrinsic, intrinsic_weight)
    adv = np.empty_like(v)
    vt = np.empty_like(v) if use_gae else None
    boot = np.asarray(bootstrap, np.float64)
    for m in range(v.shape[1]):
        for s, e, last_r in fragments(d[:, m], boot[m]):
            a, t = compute_advantages_fragment(r[s:e, m], v[s:e, m], last_r, gamma, lambda_, use_gae)
            adv[s:e, m] = a
            if use_gae:
                vt[s:e, m] = t
    return adv, vt


def vtrace_fragment(log_rhos, rewards, values, bootstrap_value, gamma, clip_rho_threshold, clip_pg_rho_threshold):
    """vtrace.from_importance_weights on one fragment, discounts = gamma, literally -> (vs, pg_advantages)."""
    rhos = np.exp(log_rhos)
    clipped_rhos = np.minimum(clip_rho_threshold, rhos)
    cs = np.minimum(1.0, rhos)
    values_t_plus_1 = np.concatenate([values[1:], [bootstrap_value]])
    deltas = clipped_rhos * (rewards + gamma * values_t_plus_1 - values)
    vs_minus_v_xs = np.empty_like(values)
    acc = 0.0
    for t in range(len(values) - 1, -1, -1):
        acc = deltas[t] + gamma * cs[t] * acc
        vs_minus_v_xs[t] = acc
    vs = vs_minus_v_xs + values
    vs_t_plus_1 = np.concatenate([vs[1:], [bootstrap_value]])
    clipped_pg_rhos = np.minimum(clip_pg_rho_threshold, rhos)
    return vs, clipped_pg_rhos * (rewards + gamma * vs_t_plus_1 - values)


def vtrace(rewards, values, dones, bootstrap, target_logp, behaviour_logp, gamma, clip_rho_threshold, clip_pg_rho_threshold,
           intrinsic=None, intrinsic_weight=0.0):
    """[T, M] float64 vs and pg_advantages of every column, fragment by fragment."""
    r, v, d = _columns(rewards, values, dones, intrinsic, intrinsic_weight)
    log_rhos = np.asarray(target_logp, np.float64) - np.asarray(behaviour_logp, np.float64)
    vs, pg = np.empty_like(v), np.empty_like(v)
    boot = np.asarray(bootstrap, np.float64)
    for m in range(v.shape[1]):
        for s, e, last_r in fragments(d[:, m], boot[m]):
            vs[s:e, m], pg[s:e, m] = vtrace_fragment(log_rhos[s:e, m], r[s:e, m], v[s:e, m], last_r, gamma, clip_rho_threshold,
                                                     clip_pg_rho_threshold)
    return vs, pg


def error_bound(mode, rewards, values, dones, bootstrap, gamma, lambda_=1.0, intrinsic=None, intrinsic_weight=0.0, target_logp=None,
                behaviour_logp=None, clip_rho_threshold=np.inf, clip_pg_rho_threshold=np.inf):
    """Elementwise bounds (out0, out1 or None) on |fp32 result - float64 result| for mode 'gae', 'returns' or 'vtrace'.

    Each step of the fp32 recurrence rounds at most c = 10 + max |log rho| times (the reward and its intrinsic term, gamma V, the
    two subtractions, rho_bar and c from expf -- whose argument carries |log rho| u of its own --, k acc and the sum, and, on the
    chunked path, the chunk's K and the carry), each a relative error of at most u = 2^-24 of a quantity bounded by the same
    recurrence run on magnitudes, A_t = a_t + k_t A_{t+1} (a_t = |x_t| with every term taken absolutely).  An error made at step
    s reaches step t scaled by k_t..k_{s-1} <= 1, so the error of acc_t is at most c (T - t + 1) u A_t; value targets and vs add
    |V_t|, pg_advantages rho_pg_t (|r_t| + gamma (A_{t+1} + |V_{t+1}|) + |V_t|)."""
    r, v, d = _columns(rewards, values, dones, intrinsic, intrinsic_weight)
    r_abs = np.abs(np.asarray(rewards, np.float64))
    if intrinsic is not None:
        r_abs = r_abs + abs(float(intrinsic_weight)) * np.abs(np.asarray(intrinsic, np.float64))
    v_abs = np.abs(v)
    t_count = v.shape[0]
    boot = np.abs(np.asarray(bootstrap, np.float64))
    c = 10.0
    rho = rho_bar = rho_pg = np.ones_like(v)
    k = np.full_like(v, gamma * lambda_ if mode == "gae" else gamma)
    if mode == "vtrace":
        log_rho = np.asarray(target_logp, np.float64) - np.asarray(behaviour_logp, np.float64)
        c += float(np.abs(log_rho).max())
        rho = np.exp(log_rho)
        rho_bar, rho_pg = np.minimum(clip_rho_threshold, rho), np.minimum(clip_pg_rho_threshold, rho)
        k = gamma * np.minimum(1.0, rho)
    big_a = np.empty_like(v)
    acc = boot.copy() if mode == "returns" else np.zeros_like(boot)
    vn = boot.copy()
    pg = np.empty_like(v)
    for t in range(t_count - 1, -1, -1):
        done = d[t]
        vn_t = np.where(done, 0.0, vn)
        acc_next = np.where(done, 0.0, acc)
        if mode == "returns":
            a = r_abs[t]
        else:
            a = rho_bar[t] * (r_abs[t] + gamma * vn_t + v_abs[t])
        pg[t] = rho_pg[t] * (r_abs[t] + gamma * (acc_next + vn_t) + v_abs[t])
        acc = a + k[t] * acc_next
        big_a[t] = acc
        vn = v_abs[t]
    steps = (t_count - np.arange(t_count) + 1.0)[:, None]
    tol = c * steps * U
    if mode == "returns":
        return tol * big_a, None
    if mode == "gae":
        return tol * big_a, tol * (big_a + v_abs)
    return tol * (big_a + v_abs), tol * pg
