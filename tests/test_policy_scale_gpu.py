"""The policy kernels at the sizes training runs them, against references that share no code with them.

The trunk (csrc/ssd_policy.cu) and the fused head (csrc/ssd_policy_head.cu) run persistent grids of at most #SMs CTAs, 128
agents per group.  At 65 536 Harvest envs x 5 agents a CTA runs ~17 groups: the accumulators and barrier parities that
alternate per group, the observation double buffer, the image-row ring carried across groups and the head's per-group
barrier are exercised only when a CTA runs several groups, so every size here is chosen so that each CTA runs at least four,
and each test asserts that premise.

  float64 reference   a float64 torch restatement of trunk, LSTM and heads on the device (pinned to oracle/policy_ref.py to
                      1e-10 on 4 096 rows), three recurrent steps from a random state, every row within the tolerances of
                      test_policy_gpu.py: shared weights (random pixels and 327 680 Harvest agents), per-agent weights;
  decomposition       an agent's result does not depend on which CTA ran it or at which group ordinal: one call at the large
                      size == the concatenation of calls that run one group per CTA, bitwise;
  sampling            the Gumbel-max sampler against a host Philox4x32-10 (numpy, pinned to oracle/philox_ref.py): with all
                      logits exactly 0 the action is the first argmax of the words' top 24 bits, tolerance-free; with random
                      logits the float64 argmax of logit + Gumbel wherever its margin exceeds 1e-3; 1..15 outputs, shared /
                      per-agent / pool, seeds with all key bits in use;
  lstm cell           ssd_policy_lstm_cell (the unfused route's cell update) against float64 from the same bf16 gates;
  alignment           the Python wrappers copy views that do not start on the 16-byte boundary the C ABI requires."""
import ctypes as C

import numpy as np
import pytest
import torch

from test_policy_gpu import FWD_TOL, TRUNK_TOL

pytestmark = pytest.mark.gpu

GA = 128                                 # agents per group of both fused kernels
HARVEST_ENVS, HARVEST_AGENTS = 65536, 5
SCALE_M = HARVEST_ENVS * HARVEST_AGENTS  # 327 680 agents: the batch the project is measured on
PIN_TOL = 1e-10                          # device float64 reference vs the numpy float64 oracle


def _policy():
    from sequential_social_dilemma_games_b200 import policy
    return policy


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _groups(m):
    return (m + GA - 1) // GA


def _maxerr(got, want):
    return (got.double() - want).abs().max().item()


@pytest.fixture(scope="module")
def harvest_obs():
    """Three consecutive observation tensors of 65 536 Harvest envs x 5 agents from the step kernel, [327 680, 15, 15, 3]."""
    from sequential_social_dilemma_games_b200.batched import BatchedSSDEnv, make_config
    cfg = make_config("harvest", num_agents=HARVEST_AGENTS)
    env = BatchedSSDEnv(cfg, HARVEST_ENVS, seed=17)
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(17)
    out = []
    for _ in range(3):
        a = torch.randint(0, cfg.num_actions, (HARVEST_ENVS, HARVEST_AGENTS), dtype=torch.int8, device="cuda", generator=g)
        obs, _ = env.step(a)
        out.append(obs.reshape(-1, 15, 15, 3).clone())
    torch.cuda.synchronize()
    env.close()
    return out


def _random_obs(m, seed, steps=3):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randint(0, 256, (m, 15, 15, 3), dtype=torch.uint8, device="cuda", generator=g) for _ in range(steps)]


def _random_state(m, seed, u=128):
    """h in [-1, 1], c in [-3, 3], agent-major fp32 rows."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    h = torch.rand((m, u), device="cuda", generator=g) * 2 - 1
    c = torch.rand((m, u), device="cuda", generator=g) * 6 - 3
    return h, c


# ---------------------------------------------------------------------------------------------------- float64 reference
def _w64(w):
    return {k: torch.from_numpy(np.asarray(v, np.float64)).cuda() for k, v in w.items()}


def features64(t, obs, chunk=1 << 15):
    """oracle/policy_ref.features on the device: uint8 [M, 15, 15, 3] -> float64 [M, 32], in chunks of rows (t = _w64(w))."""
    k = t["conv_w"].permute(3, 2, 0, 1)                                  # [kh, kw, in, out] -> [out, in, kh, kw]
    out = torch.empty((obs.shape[0], 32), dtype=torch.float64, device=obs.device)
    for a in range(0, obs.shape[0], chunk):
        x = ((obs[a:a + chunk].to(torch.float64) - 128.0) / 255.0).permute(0, 3, 1, 2)
        y = torch.relu(torch.nn.functional.conv2d(x, k, t["conv_b"])).permute(0, 2, 3, 1).reshape(x.shape[0], -1)
        y = torch.relu(y @ t["fc1_w"] + t["fc1_b"])
        out[a:a + chunk] = torch.relu(y @ t["fc2_w"] + t["fc2_b"])
    return out


def step64(t, x, h, c):
    """oracle/policy_ref.forward after the trunk, on the device: -> (logits, value, h', c'), float64."""
    z = x @ t["lstm_w"] + h @ t["lstm_u"] + t["lstm_b"]
    zi, zf, zc, zo = z.chunk(4, dim=1)
    c2 = torch.sigmoid(zf) * c + torch.sigmoid(zi) * torch.tanh(zc)
    h2 = torch.sigmoid(zo) * torch.tanh(c2)
    return h2 @ t["logits_w"] + t["logits_b"], (h2 @ t["value_w"] + t["value_b"])[:, 0], h2, c2


def _pin_rows(m, n=4096, seed=0):
    """Up to n rows of [0, m): the first and last row of 64 groups spread over the batch, the ragged tail, random rows."""
    g = np.unique(np.linspace(0, _groups(m) - 1, 64).astype(np.int64))
    edge = np.unique(np.concatenate([g * GA, np.minimum(g * GA + GA - 1, m - 1), np.arange(max(0, m - 2 * GA), m)]))
    rest = np.setdiff1d(np.random.RandomState(seed).permutation(m)[:n], edge)[:max(0, n - len(edge))]
    return np.sort(np.concatenate([edge, rest]))


class Reference64(object):
    """The network in float64 on the device, agent m evaluated with sets[m % P] (the agent-major column of a [B, P] batch),
    carrying its own (h, c) from the given fp32 rows."""

    def __init__(self, sets, h0, c0):
        self.sets, self.t = sets, [_w64(w) for w in sets]
        m = h0.shape[0]
        self.cols = [torch.arange(p, m, len(sets), device="cuda") for p in range(len(sets))]
        self.h, self.c = h0.double(), c0.double()

    def step(self, obs):
        obs = obs.reshape(-1, 15, 15, 3)
        m, A = obs.shape[0], self.sets[0]["logits_w"].shape[1]
        x = torch.empty((m, 32), dtype=torch.float64, device="cuda")
        lg = torch.empty((m, A), dtype=torch.float64, device="cuda")
        v = torch.empty((m,), dtype=torch.float64, device="cuda")
        h, c = torch.empty_like(self.h), torch.empty_like(self.c)
        for t, r in zip(self.t, self.cols):
            x[r] = features64(t, obs[r])
            lg[r], v[r], h[r], c[r] = step64(t, x[r], self.h[r], self.c[r])
        self.h, self.c = h, c
        return x, lg, v, h, c

    def pin(self, obs, h_prev, c_prev, out, rows):
        """`out` (a step from (h_prev, c_prev)) == oracle/policy_ref.py on `rows`, to PIN_TOL."""
        from oracle import policy_ref
        P = len(self.sets)
        obs = obs.reshape(-1, 15, 15, 3)
        for p in range(P):
            r = rows[rows % P == p]
            rt = torch.from_numpy(r).cuda()
            on = obs[rt].cpu().numpy()
            want = (policy_ref.features(self.sets[p], on),) + policy_ref.forward(self.sets[p], on, h_prev[rt].cpu().numpy(), c_prev[rt].cpu().numpy())
            for name, got, w in zip(("features", "logits", "value", "h", "c"), out, want):
                err = np.abs(got[rt].cpu().numpy() - w).max()
                assert err < PIN_TOL, (name, p, err)


def _check_forward_at_scale(sets, steps, seed):
    """Three recurrent steps of the kernels (from a random state) against Reference64, every row; the reference is pinned to the
    numpy oracle on the first step."""
    policy = _policy()
    P = len(sets)
    net = policy.ConvToFCNet(sets if P > 1 else sets[0])
    m = steps[0].numel() // (15 * 15 * 3)
    h0, c0 = _random_state(m, seed)
    ref = Reference64(sets, h0, c0)
    h, c = net.state_from_rows(h0), net.state_from_rows(c0)
    for t, obs in enumerate(steps):
        h_prev, c_prev = ref.h, ref.c
        want = ref.step(obs)
        if t == 0:
            ref.pin(obs, h_prev, c_prev, want, _pin_rows(m, seed=seed))
        feats = net.features(obs)
        logits, value, h, c = net.forward(obs, h, c)
        err = _maxerr(feats, want[0])
        assert err < TRUNK_TOL, (t, "features", err)
        for name, got, w in zip(("logits", "value", "h", "c"), (logits, value, net.state_rows(h, m), net.state_rows(c, m)), want[1:]):
            err = _maxerr(got, w)
            assert err < FWD_TOL, (t, name, err)
    assert want[1].abs().max().item() > 0.1 and want[4].abs().max().item() > 1.0   # not vacuous
    net.close()


@pytest.mark.parametrize("source", ["random", "harvest"])
def test_shared_net_matches_float64_at_scale(source, harvest_obs):
    """Shared weights at 4 sms 128 + 77 random-pixel agents and at 65 536 Harvest envs x 5 agents."""
    sms = _sms()
    steps = _random_obs(4 * sms * GA + 77, seed=31) if source == "random" else harvest_obs
    m = steps[0].shape[0]
    assert _groups(m) >= 4 * sms   # every CTA runs at least four groups
    _check_forward_at_scale([_policy().random_weights(num_outputs=8, seed=41)], steps, seed=51)


@pytest.mark.parametrize("P,tail", [(5, 77), (16, 5)])
def test_per_agent_net_matches_float64_at_scale(P, tail):
    """Per-agent weights: B = 4 floor(sms / P) 128 + tail envs of P agents (P floor(sms / P) CTAs, one policy each)."""
    sms = _sms()
    B = 4 * (sms // P) * GA + tail
    assert _groups(B) >= 4 * (sms // P)   # every CTA of a policy runs at least four groups
    g = torch.Generator(device="cuda").manual_seed(P)
    steps = [torch.randint(0, 256, (B, P, 15, 15, 3), dtype=torch.uint8, device="cuda", generator=g) for _ in range(3)]
    sets = [_policy().random_weights(num_outputs=8, seed=600 + p) for p in range(P)]
    _check_forward_at_scale(sets, steps, seed=P)


# ---------------------------------------------------------------------------------------------------- decomposition
def test_shared_net_result_does_not_depend_on_cta_or_group_ordinal():
    """One call at 4 sms 128 + 77 agents (every CTA runs 4-5 groups) == calls over slices of sms 128 agents (one group per CTA),
    bitwise: features, logits, value, h', c'."""
    policy = _policy()
    sms = _sms()
    m, cut = 4 * sms * GA + 77, sms * GA
    assert _groups(m) >= 4 * sms and _groups(cut) == sms
    net = policy.ConvToFCNet(policy.random_weights(num_outputs=8, seed=43))
    obs = _random_obs(m, seed=43, steps=1)[0]
    h0, c0 = _random_state(m, seed=43)
    h, c = net.state_from_rows(h0), net.state_from_rows(c0)
    whole = (net.features(obs),) + net.forward(obs, h, c)
    parts = []
    for a in range(0, m, cut):
        ga, gb = a // GA, _groups(min(a + cut, m))
        parts.append((net.features(obs[a:a + cut]),) + net.forward(obs[a:a + cut], h[ga:gb], c[ga:gb]))
    for i, name in enumerate(("features", "logits", "value")):
        assert torch.equal(whole[i], torch.cat([p[i] for p in parts])), name
    for i, name in ((3, "h"), (4, "c")):
        rows = torch.cat([net.state_rows(p[i], min(cut, m - k * cut)) for k, p in enumerate(parts)])
        assert torch.equal(net.state_rows(whole[i], m), rows), name
    net.close()


@pytest.mark.parametrize("P,tail", [(5, 77), (16, 5)])
def test_per_agent_result_does_not_depend_on_cta_or_group_ordinal(P, tail):
    """Per-agent weights: one call at B = 4 floor(sms / P) 128 + tail == calls over slices of floor(sms / P) 128 envs along B
    (one group per CTA), bitwise; the state is cut through state_rows / state_from_rows."""
    policy = _policy()
    sms = _sms()
    B, cut = 4 * (sms // P) * GA + tail, (sms // P) * GA
    assert _groups(B) >= 4 * (sms // P) and _groups(cut) == sms // P
    net = policy.ConvToFCNet([policy.random_weights(num_outputs=8, seed=700 + p) for p in range(P)])
    g = torch.Generator(device="cuda").manual_seed(7)
    obs = torch.randint(0, 256, (B, P, 15, 15, 3), dtype=torch.uint8, device="cuda", generator=g)
    h0, c0 = _random_state(B * P, seed=7)
    whole = (net.features(obs),) + net.forward(obs, net.state_from_rows(h0), net.state_from_rows(c0))
    parts = []
    for a in range(0, B, cut):
        b = min(a + cut, B)
        hs, cs = net.state_from_rows(h0[a * P:b * P]), net.state_from_rows(c0[a * P:b * P])
        f = net.features(obs[a:b])
        lg, v, h2, c2 = net.forward(obs[a:b], hs, cs)
        parts.append((f, lg, v, net.state_rows(h2, (b - a) * P), net.state_rows(c2, (b - a) * P)))
    for i, name in enumerate(("features", "logits", "value")):
        assert torch.equal(whole[i], torch.cat([p[i] for p in parts])), name
    assert torch.equal(net.state_rows(whole[3], B * P), torch.cat([p[3] for p in parts])), "h"
    assert torch.equal(net.state_rows(whole[4], B * P), torch.cat([p[4] for p in parts])), "c"
    net.close()


# ---------------------------------------------------------------------------------------------------- sampling
_M0, _M1, _W0, _W1, _MASK = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85, 0xFFFFFFFF


def philox4x32_10_np(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 over uint32 arrays (broadcast): counters (c0, c1, c2, c3), key (k0, k1) scalars -> uint32 [..., 4]."""
    mask, s = np.uint64(_MASK), np.uint64(32)
    c0, c1, c2, c3 = np.broadcast_arrays(*[np.asarray(x, np.uint64) & mask for x in (c0, c1, c2, c3)])
    k0, k1 = np.uint64(k0 & _MASK), np.uint64(k1 & _MASK)
    for _ in range(10):
        p0, p1 = c0 * np.uint64(_M0), c2 * np.uint64(_M1)   # < 2^64: exact in uint64
        c0, c1, c2, c3 = (p1 >> s) ^ c1 ^ k0, p1 & mask, (p0 >> s) ^ c3 ^ k1, p0 & mask
        k0, k1 = (k0 + np.uint64(_W0)) & mask, (k1 + np.uint64(_W1)) & mask
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def test_numpy_philox_matches_oracle():
    """philox4x32_10_np == oracle/philox_ref.philox4x32_10 on 300 counters and keys, key words with the high bit set included."""
    from oracle import philox_ref
    rng = np.random.RandomState(0)
    ctr = rng.randint(0, 2 ** 32, size=(300, 4), dtype=np.uint64)
    ctr[:8] = [[0, 0, 0, 0], [_MASK] * 4, [1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 0], [0, 0, 0, 1], [65536, 0, 2, 3], [2 ** 31, 2 ** 31, 0, 0]]
    keys = rng.randint(0, 2 ** 32, size=(300, 2), dtype=np.uint64)
    keys[:100] |= np.uint64(0x80000000)
    keys[100:110] = [[_MASK, _MASK], [0, 0], [7, 1], [0x80000000, 0], [0, 0x80000000], [1, 2], [_MASK, 0], [0, _MASK], [3, 3], [2 ** 31 - 1, 2 ** 31]]
    for (c, k) in zip(ctr, keys):
        got = philox4x32_10_np(c[0], c[1], c[2], c[3], int(k[0]), int(k[1]))
        assert tuple(int(x) for x in got) == philox_ref.philox4x32_10(tuple(int(x) for x in c), (int(k[0]), int(k[1])))
    # vectorised over the counter equals element by element
    batch = philox4x32_10_np(ctr[:, 0], ctr[:, 1], ctr[:, 2], ctr[:, 3], 0xDEADBEEF, 0x80000001)
    for i in range(0, 300, 37):
        assert tuple(int(x) for x in batch[i]) == philox_ref.philox4x32_10(tuple(int(x) for x in ctr[i]), (0xDEADBEEF, 0x80000001))


def sampler_words(seed, counter, m, A):
    """The words the head's sampler draws for agents m (int64 array) and outputs a < A: word a & 3 of Philox block
    (m lo, m hi, counter, a >> 2) under key (seed lo, seed hi) -> uint32 [len(m), A]."""
    m = np.asarray(m, np.uint64)
    blocks = [philox4x32_10_np(m, m >> np.uint64(32), counter, b, seed & _MASK, seed >> 32) for b in range((A + 3) // 4)]
    return np.concatenate(blocks, axis=1)[:, :A]


def _uniform(words):
    """u = ((w >> 8) + 0.5) 2^-24, exactly (float64)."""
    return ((words >> 8).astype(np.float64) + 0.5) * 2.0 ** -24


SEEDS = [0, 2 ** 32 + 7, 2 ** 64 - 1]
NEAR_ONE = 1 - 2.0 ** -20


def _sample_rows(m, seed):
    """Agents a sampled check covers when it cannot afford all: both ends, either side of 2^16 (where a key truncated to 16
    bits of m starts to repeat), and random agents."""
    rng = np.random.RandomState(seed)
    pick = [np.arange(0, 2048), np.arange(65536 - 1024, 65536 + 1024), np.arange(m - 2048, m), rng.choice(m, 32768, replace=False)]
    return np.unique(np.concatenate(pick))


def _check_zero_logit_draws(actions, words):
    """All logits are 0: the action is the first argmax over a of w_a >> 8.  Agents whose two largest u lie within 2^-12 of each
    other are left out (the kernel's fast logarithms may order them either way).  -> (agents left out, near-one draws checked)."""
    k = (words >> 8).astype(np.int64)
    want = k.argmax(axis=1)   # first maximum
    if k.shape[1] > 1:
        top2 = np.sort(k, axis=1)[:, -2:]
        ok = (top2[:, 1] - top2[:, 0]) * 2.0 ** -24 > 2.0 ** -12
    else:
        ok = np.ones(k.shape[0], bool)
    bad = np.flatnonzero(ok & (actions != want))
    assert bad.size == 0, ("zero logits: %d agents differ" % bad.size, bad[:8], actions[bad[:8]], want[bad[:8]],
                           _uniform(words[bad[:8]]))
    near = (_uniform(words) >= NEAR_ONE).any(axis=1)
    return int((~ok).sum()), int((near & ok).sum())


def _check_gumbel_argmax(actions, logits, words, live):
    """Random logits: the kernel's action == argmax_a(logit_a - log(-log u_a)) in float64 from the kernel's own fp32 logits,
    for every agent whose top-two score margin exceeds 1e-3.  -> number of agents left out."""
    g = -np.log(-np.log(_uniform(words)))
    s = logits.astype(np.float64) + g
    want = s.argmax(axis=1)
    if s.shape[1] > 1:
        top2 = np.sort(s, axis=1)[:, -2:]
        ok = top2[:, 1] - top2[:, 0] > 1e-3
    else:
        ok = np.ones(s.shape[0], bool)
    ok &= live
    bad = np.flatnonzero(ok & (actions != want))
    assert bad.size == 0, ("random logits: %d agents differ" % bad.size, bad[:8], actions[bad[:8]], want[bad[:8]])
    return int((live & ~ok).sum())


def _sampling_net(kind, A, zero_logits=False):
    """(net, P, ids) of one kind at 327 680 agents: shared weights, per-agent (P = 5) or a pool of K = 7 with ~1 % skipped ids."""
    policy = _policy()
    n_sets = {"shared": 1, "per_agent": HARVEST_AGENTS, "pool": 7}[kind]
    sets = [policy.random_weights(num_outputs=A, seed=900 + 10 * A + k) for k in range(n_sets)]
    for w in sets:
        if zero_logits:
            w["logits_w"][:] = 0
            w["logits_b"][:] = 0
        else:
            w["logits_b"] = np.linspace(-1, 1, A).astype(np.float32)
    if kind == "shared":
        return policy.ConvToFCNet(sets[0]), None
    if kind == "per_agent":
        return policy.ConvToFCNet(sets), None
    g = torch.Generator(device="cuda").manual_seed(A)
    ids = torch.randint(0, n_sets, (SCALE_M,), dtype=torch.uint8, device="cuda", generator=g)
    skip = torch.rand((SCALE_M,), device="cuda", generator=g) < 0.01
    ids[skip] = torch.randint(n_sets, 256, (int(skip.sum()),), dtype=torch.uint8, device="cuda", generator=g)
    return policy.PolicyPool(sets), ids


def _act(net, ids, obs, h, c):
    """-> (logits, actions, h', c') of one sampling call, logits as the kernel computed them for its draws."""
    if ids is None:
        logits, _, h, c, a = net._fused(obs, h, c, sample=True)
    else:
        logits, _, h, c, a = net._run(obs, ids, h, c, sample=True)
    return logits, a, h, c


@pytest.mark.parametrize("A", [1, 2, 4, 5, 8, 15])
def test_sampling_with_zero_logits_is_the_argmax_of_the_philox_words(A, harvest_obs):
    """Every logit is exactly 0, so the sampled action depends on the Philox words alone: the first argmax over a of w_a >> 8,
    for every agent of 327 680, three consecutive calls and three seeds (all 64 key bits in use); seeding again repeats the
    first call.  Draws with u >= 1 - 2^-20 are among those checked."""
    net, _ = _sampling_net("shared", A, zero_logits=True)
    m = SCALE_M
    assert _groups(m) >= 4 * _sms()
    agents = np.arange(m)
    left_out = near = 0
    for seed in SEEDS:
        net.seed_sampling(seed)
        h, c = net.initial_state(m)
        first = None
        for call, obs in enumerate(harvest_obs):
            logits, a, h, c = _act(net, None, obs, h, c)
            if call == 0:
                assert not logits.any()
                first = a
            lo, nr = _check_zero_logit_draws(a.long().cpu().numpy(), sampler_words(seed, call, agents, A))
            left_out, near = left_out + lo, near + nr
        net.seed_sampling(seed)
        assert torch.equal(_act(net, None, harvest_obs[0], *net.initial_state(m))[1], first)
    assert left_out < 0.01 * 9 * m, left_out
    if 9 * m * A * 2.0 ** -20 >= 10:   # expected number of draws with u >= 1 - 2^-20 (at least 10 from A = 4 on)
        assert near > 0
    net.close()


@pytest.mark.parametrize("A", [1, 2, 4, 5, 8, 15])
@pytest.mark.parametrize("kind", ["shared", "per_agent", "pool"])
def test_sampling_with_random_logits_matches_float64_gumbel_argmax(kind, A, harvest_obs):
    """The kernel's action == the float64 Gumbel-max of its own logits and the host Philox draws wherever the margin exceeds
    1e-3, at 327 680 agents (every agent on a seed's first call, 38 912 of them on the next two), three seeds; the pool's
    skipped agents get -1."""
    net, ids = _sampling_net(kind, A)
    m = SCALE_M
    obs_steps = [o.reshape(HARVEST_ENVS, HARVEST_AGENTS, 15, 15, 3) for o in harvest_obs] if kind == "per_agent" else harvest_obs
    live = np.ones(m, bool) if ids is None else ids.cpu().numpy() < net.num_policies
    if ids is not None:
        assert 0.005 < 1 - live.mean() < 0.02
    left_out = checked = 0
    for seed in SEEDS:
        net.seed_sampling(seed)
        h, c = net.initial_state(m)
        first = None
        for call, obs in enumerate(obs_steps):
            logits, a, h, c = _act(net, ids, obs, h, c)
            a = a.long().cpu().numpy()
            first = a if call == 0 else first
            assert (a[~live] == -1).all() and (a[live] >= 0).all() and (a[live] < A).all()
            rows = np.arange(m) if call == 0 else _sample_rows(m, seed=call)
            left_out += _check_gumbel_argmax(a[rows], logits.cpu().numpy()[rows], sampler_words(seed, call, rows, A), live[rows])
            checked += int(live[rows].sum())
        net.seed_sampling(seed)
        h, c = net.initial_state(m)
        assert np.array_equal(_act(net, ids, obs_steps[0], h, c)[1].long().cpu().numpy(), first)
    assert left_out < 0.02 * checked, (left_out, checked)
    net.close()


# ---------------------------------------------------------------------------------------------------- lstm cell
@pytest.mark.parametrize("M", ["1", "3", "1000", "4*sms*128+1"])
@pytest.mark.parametrize("units", [8, 24, 128, 256])
def test_lstm_cell_matches_float64(units, M):
    """ssd_policy_lstm_cell: c' and h' within 1e-5 of float64 computed from the same bf16 gates, bias and c; h' as bf16 ==
    h'.to(bfloat16), bitwise.  M u / 8 threads: shapes that leave a partial last block of 256 included."""
    from sequential_social_dilemma_games_b200 import _lib
    m = {"1": 1, "3": 3, "1000": 1000}.get(M) or 4 * _sms() * GA + 1
    g = torch.Generator(device="cuda").manual_seed(units * 7 + m)
    gates = (torch.randn((m, 4 * units), device="cuda", generator=g) * 3).to(torch.bfloat16)
    bias = torch.randn((4 * units,), device="cuda", generator=g)
    c = torch.rand((m, units), device="cuda", generator=g) * 6 - 3
    c_out, h_out = torch.empty_like(c), torch.empty_like(c)
    h16 = torch.empty((m, units), dtype=torch.bfloat16, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert _lib.lib.ssd_policy_lstm_cell(p(gates), p(bias), p(c), p(c_out), p(h_out), p(h16), m, units, st) == 0
    z = gates.double() + bias.double()
    zi, zf, zc, zo = z.chunk(4, dim=1)
    c64 = torch.sigmoid(zf) * c.double() + torch.sigmoid(zi) * torch.tanh(zc)
    h64 = torch.sigmoid(zo) * torch.tanh(c64)
    assert _maxerr(c_out, c64) < 1e-5, _maxerr(c_out, c64)
    assert _maxerr(h_out, h64) < 1e-5, _maxerr(h_out, h64)
    assert torch.equal(h16, h_out.to(torch.bfloat16))
    if m * units >= 8000:   # not vacuous: large cell states and outputs occur
        assert c64.abs().max().item() > 2.0 and h64.abs().max().item() > 0.5


# ---------------------------------------------------------------------------------------------------- alignment
def _misaligned_copy(t):
    """A contiguous copy of t whose data starts 4 bytes past a 16-byte boundary."""
    buf = torch.empty((t.numel() * t.element_size() + 16,), dtype=torch.uint8, device=t.device)
    v = buf[4:4 + t.numel() * t.element_size()].view(t.dtype).view(t.shape)
    v.copy_(t)
    assert v.is_contiguous() and v.data_ptr() % 16 != 0
    return v


def _assert_same_step(net, m, got, want):
    """(logits, value, h', c') equal bitwise; the state compared as agent rows (the padding rows of the tiled layout are not written)."""
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    for g, w in zip(got[2:], want[2:]):
        assert torch.equal(net.state_rows(g, m), net.state_rows(w, m))


@pytest.mark.parametrize("k", [1, 3, 127])
def test_views_off_the_16_byte_boundary_are_copied(k):
    """features(obs[k:]) == features(obs)[k:] bitwise (shared, per-agent, pool): obs[k:] is contiguous but starts 675 k bytes in;
    a recurrent state that starts off the boundary gives what the aligned one gives (fused, unfused and pool routes)."""
    policy = _policy()
    m = 1000
    obs = _random_obs(m, seed=k, steps=1)[0]
    w = policy.random_weights(num_outputs=8, seed=k)
    net = policy.ConvToFCNet(w)
    assert obs[k:].is_contiguous() and obs[k:].data_ptr() % 16 != 0
    assert torch.equal(net.features(obs[k:]), net.features(obs)[k:])
    h, c = net.state_from_rows(_random_state(m, seed=k)[0]), net.state_from_rows(_random_state(m, seed=k)[1])
    _assert_same_step(net, m, net.forward(obs, _misaligned_copy(h), _misaligned_copy(c)), net.forward(obs, h, c))
    net.close()
    per = policy.ConvToFCNet([policy.random_weights(num_outputs=8, seed=k + p) for p in range(5)])
    obs5 = obs[:1000 // 5 * 5].reshape(-1, 5, 15, 15, 3)
    assert torch.equal(per.features(obs5[k:]), per.features(obs5)[5 * k:])
    per.close()
    pool = policy.PolicyPool([policy.random_weights(num_outputs=8, seed=k + p) for p in range(3)])
    ids = torch.randint(0, 3, (m,), dtype=torch.uint8, device="cuda", generator=torch.Generator(device="cuda").manual_seed(k))
    assert torch.equal(pool.features(obs[k:], ids[k:]), pool.features(obs, ids)[k:])
    hp, cp = pool.state_from_rows(_random_state(m, seed=k)[0]), pool.state_from_rows(_random_state(m, seed=k)[1])
    _assert_same_step(pool, m, pool.forward(obs, ids, _misaligned_copy(hp), _misaligned_copy(cp)), pool.forward(obs, ids, hp, cp))
    pool.close()
    small = policy.ConvToFCNet(policy.random_weights(num_outputs=8, cell_size=24, seed=k))
    hs, cs = _random_state(m, seed=k, u=24)
    _assert_same_step(small, m, small.forward(obs, hs, _misaligned_copy(cs)), small.forward(obs, hs, cs))
    small.close()
