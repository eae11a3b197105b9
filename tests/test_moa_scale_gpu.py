"""The MOA kernel (csrc/ssd_policy_moa.cu) at the sizes training runs it, against a float64 reference that shares no code with it.

The kernel runs persistent grids of at most #SMs CTAs, 128 agents per group (Shared, PerAgent) or per tile of one weight set
(Pool).  Tensor memory, the mbarrier parity, the scratch and, for the pool, the resident weight set are carried from one group
to the next, so every case here runs at least four groups or tiles per CTA and asserts that premise.

  MOAReference64   a float64 torch restatement of oracle/moa_ref.py on the device, in chunks of rows: the input is built
                   literally as [x | onehot(own) | onehot(others)] (zero rows for invalid actions) with one matmul per own
                   action a', not with the kernel's row-gather algebra; agent m uses weight set m % N (per-agent) or ids[m]
                   (pool).  It is pinned to oracle/moa_ref.moa_forward to 1e-10 on at most ~4 096 rows chosen by the kernel's
                   group map (the first and last rows of groups spread over the batch, the ragged tail, every row of an env
                   with an invalid action, random rows), for KL, JSD and a clip.
  every row        three recurrent steps from a random state: pred, counterfactual, h' and c' within MOA_TOL; influence and
                   influence_per_agent within OWN_TOL (1 + |v|) of float64 recomputed from the kernel's own pred,
                   counterfactual and policy logits, and within the end-to-end bound of test_moa_gpu.py of the reference;
                   influence, pred, h' and c' bitwise the same with counterfactuals on and off.
  cases            shared weights on closed-loop Harvest inputs (65 536 envs x 5 agents); per-agent weights (5, 8) on the same
                   inputs, (5, 9) and (16, 4) on random inputs; the pool at K = 40 with ~1 % skipped ids (their rows keep the
                   values the caller wrote) and at K = 255 with every CTA crossing a weight-set boundary; invalid actions in
                   ~0.1 % of envs, at group boundaries and in the ragged tail, for A = 8 and A = 9 (the extra drain of an
                   invalid own action runs on the first or the second half of the CTA).

Every call goes through the C ABI with sentinel-filled outputs, so a row the kernel does not write is seen as such, and the
joint actions reach the kernel as given (127 and -128 included; MOANet.step would clamp them to A and -1).  The largest error
against each tolerance is recorded as a test property (pytest --junitxml)."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from test_moa_gpu import MOA_TOL, OWN_TOL, _inputs, _weights
from test_policy_scale_gpu import GA, HARVEST_AGENTS, HARVEST_ENVS, PIN_TOL, _random_state

pytestmark = pytest.mark.gpu

SENTINELS = {"pred": 7.5, "counterfactual": -7.5, "influence_per_agent": 9.5, "influence": -9.5, "h": 3.25, "c": -3.25}


def _policy():
    from sequential_social_dilemma_games_b200 import policy
    return policy


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _cdiv(a, b):
    return -(-a // b)


# ---------------------------------------------------------------------------------------------------- float64 reference
def _w64(w):
    return {k: torch.from_numpy(np.asarray(v, np.float64)).cuda() for k, v in w.items()}


def _onehot64(a, A):
    """float64 [len(a), A]; a zero row for an action outside 0..A-1."""
    ok = (a >= 0) & (a < A)
    return torch.nn.functional.one_hot(torch.where(ok, a, torch.zeros_like(a)), A).double() * ok[:, None].double()


def _others(joint):
    """int64 [M, N-1]: for agent m = b N + i the actions a_{b, j}, j != i, in increasing j."""
    B, N = joint.shape
    m = torch.arange(B * N, device=joint.device)
    b, i = m // N, m % N
    k = torch.arange(N - 1, device=joint.device)[None, :]
    return joint.long()[b[:, None], torch.where(k < i[:, None], k, k + 1)]


def moa64(t, x, own, others, h, c, A):
    """One float64 MOA step (t = _w64(weights)) of agents with own action `own` [m] and the others' actions `others` [m, N-1]:
    -> (pred [m, N-1, A], h', c', counterfactual [m, A, N-1, A])."""
    n1 = others.shape[1]
    inp = torch.cat([x, _onehot64(own, A)] + [_onehot64(others[:, k], A) for k in range(n1)], dim=1)   # [m, 32 + N A]
    hub = h @ t["moa_lstm_u"] + t["moa_lstm_b"]

    def run(v):
        zi, zf, zc, zo = (v @ t["moa_lstm_w"] + hub).chunk(4, dim=1)
        c2 = torch.sigmoid(zf) * c + torch.sigmoid(zi) * torch.tanh(zc)
        h2 = torch.sigmoid(zo) * torch.tanh(c2)
        return (h2 @ t["moa_logits_w"] + t["moa_logits_b"]).view(-1, n1, A), h2, c2

    pred, h2, c2 = run(inp)
    cf = []
    for ap in range(A):
        v = inp.clone()
        v[:, 32:32 + A] = 0.0
        v[:, 32 + ap] = 1.0
        cf.append(run(v)[0])
    return pred, h2, c2, torch.stack(cf, dim=1)


def _kl64(p, q):
    return torch.where(p > 0, p * (torch.log(p) - torch.log(q)), torch.zeros_like(p)).sum(dim=-1)


def bad_rows(joint, A):
    """bool [M]: the agents of envs with an action outside 0..A-1."""
    return ((joint < 0) | (joint >= A)).any(dim=1).repeat_interleave(joint.shape[1])


def influence64(pred, cf, policy_logits, joint, A, divergence, clip=math.inf):
    """oracle/moa_ref.influence_from in float64 on the device: -> (influence_per_agent [M, N-1], influence [M])."""
    pi = torch.softmax(policy_logits.double(), dim=-1)
    q = torch.einsum("ma,makx->mkx", pi, torch.softmax(cf.double(), dim=-1))
    q = q / q.sum(dim=-1, keepdim=True)
    p = torch.softmax(pred.double(), dim=-1)
    if divergence == "kl":
        d = _kl64(p, q)
    else:
        mu = 0.5 * (p + q)
        d = 0.5 * _kl64(p, mu) + 0.5 * _kl64(q, mu)
    d[bad_rows(joint, A)] = math.nan
    return d, d.sum(dim=1).clamp(-clip, clip)


class MOAReference64(object):
    """The MOA in float64 on the device, agent m evaluated with sets[sel[m]] (sel >= len(sets): no MOA, rows left at zero),
    carrying its own (h, c) from the given fp32 rows."""

    def __init__(self, sets, n, a, sel, h0, c0):
        self.sets, self.t, self.n, self.a = sets, [_w64(w) for w in sets], n, a
        self.sel = sel
        self.idx = [torch.nonzero(sel == s).flatten() for s in range(len(sets))]
        self.h, self.c = h0.double(), c0.double()

    def step(self, x, joint, chunk=1 << 15):
        """-> dict pred, h, c, counterfactual of the step from the carried state, which it then replaces."""
        m, n1, A = x.shape[0], self.n - 1, self.a
        own, oth, x = joint.reshape(-1).long(), _others(joint), x.double()
        out = {"pred": torch.zeros((m, n1, A), dtype=torch.float64, device="cuda"), "h": self.h.clone(), "c": self.c.clone(),
               "counterfactual": torch.zeros((m, A, n1, A), dtype=torch.float64, device="cuda")}
        for t, r in zip(self.t, self.idx):
            for k in range(0, r.numel(), chunk):
                rr = r[k:k + chunk]
                out["pred"][rr], out["h"][rr], out["c"][rr], out["counterfactual"][rr] = moa64(t, x[rr], own[rr], oth[rr], self.h[rr],
                                                                                               self.c[rr], A)
        self.h, self.c = out["h"], out["c"]
        return out

    def pin(self, x, joint, pl, h_prev, c_prev, out, rows, divergence, clip):
        """`out` (the step from (h_prev, c_prev), with its influence for `divergence` and `clip`) == oracle/moa_ref.moa_forward
        on `rows` to PIN_TOL; NaN exactly where the oracle has NaN.  The oracle runs on whole envs (an agent's input holds its
        env's joint action) and one weight set at a time."""
        from oracle import moa_ref
        n = self.n
        sel = self.sel.cpu().numpy()
        for s, w in enumerate(self.sets):
            r = rows[sel[rows] == s]
            if not r.size:
                continue
            envs = np.unique(r // n)
            agents = (envs[:, None] * n + np.arange(n)[None, :]).reshape(-1)
            at = torch.from_numpy(agents).cuda()
            np64 = lambda v: v[at].double().cpu().numpy()
            want = moa_ref.moa_forward(w, np64(x), joint[torch.from_numpy(envs).cuda()].long().cpu().numpy(), np64(pl), np64(h_prev),
                                       np64(c_prev), self.a, divergence=divergence, clip=clip)
            pos, rt = np.searchsorted(agents, r), torch.from_numpy(r).cuda()
            for name, got in out.items():
                g, wv = got[rt].cpu().numpy(), want[name][pos]
                assert np.array_equal(np.isnan(g), np.isnan(wv)), (name, s)
                fin = ~np.isnan(wv)
                err = np.abs(g[fin] - wv[fin]).max() if fin.any() else 0.0
                assert err < PIN_TOL, (name, s, divergence, err)


def _pin_rows(edge, m, extra=(), n_rows=4096, seed=0):
    """The rows a pin covers: `edge` (group edges and ragged tail by the kernel's group map), `extra`, then random rows up to
    n_rows in all."""
    keep = np.unique(np.concatenate([np.asarray(edge, np.int64), np.asarray(extra, np.int64)]))
    rest = np.setdiff1d(np.random.RandomState(seed).permutation(m)[:n_rows], keep)[:max(0, n_rows - len(keep))]
    return np.sort(np.concatenate([keep, rest]))


def shared_edges(m):
    """Shared map: group g holds agents 128 g .. 128 g + 127; its first and last row for 64 groups spread over the batch, and
    the ragged tail (the last group)."""
    n_groups = _cdiv(m, GA)
    g = np.unique(np.linspace(0, n_groups - 1, 64).astype(np.int64))
    return np.concatenate([g * GA, np.minimum(g * GA + GA - 1, m - 1), np.arange((n_groups - 1) * GA, m)])


def per_agent_edges(B, n, groups=32):
    """Per-agent map: group g of weight set p holds agents (128 g + r) N + p, r < 128; the first and last row of `groups`
    groups spread over each set, and the ragged tail (each set's last group)."""
    n_groups = _cdiv(B, GA)
    g = np.unique(np.linspace(0, n_groups - 1, groups).astype(np.int64))
    envs = np.concatenate([g * GA, np.minimum(g * GA + GA - 1, B - 1), np.arange((n_groups - 1) * GA, B)])
    return (envs[:, None] * n + np.arange(n)[None, :]).reshape(-1)


def _live_err(got, want, live):
    """max |got - want| over live rows where want is finite (float64)."""
    d = (got.double() - want)[live]
    d = d[~torch.isnan(want[live])]
    return d.abs().max().item() if d.numel() else 0.0


# ---------------------------------------------------------------------------------------------------- kernel calls
def raw_step(net, x, ids, joint, pl, h, c, divergence, clip, counterfactuals):
    """ssd_moa_step (ids None) or ssd_moa_pool_step with sentinel-filled outputs and the int8 joint actions as given -> MOAStep."""
    from sequential_social_dilemma_games_b200 import _lib
    L = _lib.lib
    m, n, A = x.shape[0], net.num_agents, net.num_actions
    assert joint.dtype == torch.int8 and joint.is_contiguous() and joint.numel() == m
    out = {"pred": torch.full((m, n - 1, A), SENTINELS["pred"], device="cuda"),
           "counterfactual": torch.full((m, A, n - 1, A), SENTINELS["counterfactual"], device="cuda") if counterfactuals else None,
           "influence_per_agent": torch.full((m, n - 1), SENTINELS["influence_per_agent"], device="cuda"),
           "influence": torch.full((m,), SENTINELS["influence"], device="cuda"),
           "h": torch.full_like(h, SENTINELS["h"]), "c": torch.full_like(c, SENTINELS["c"])}
    p = lambda t: C.c_void_p(t.data_ptr() if t is not None else None)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    div = _lib.DIV_KL if divergence == "kl" else _lib.DIV_JSD
    io = (p(joint), p(pl), p(h), p(c), p(out["h"]), p(out["c"]), p(out["pred"]), p(out["counterfactual"]), p(out["influence_per_agent"]),
          p(out["influence"]), m, div, clip, st)
    rc = L.ssd_moa_step(net._h, p(x), *io) if ids is None else L.ssd_moa_pool_step(net._h, p(x), p(ids), *io)
    assert rc == 0, L.ssd_last_error()
    return _policy().MOAStep(out["pred"], out["influence"], out["influence_per_agent"], out["h"], out["c"], out["counterfactual"])


def _bits(t):
    return t.contiguous().view(torch.int32)


def check_at_scale(net, sets, n, a, steps, sel, edge, ids=None, divergences=("kl",), clip=math.inf, seed=0, record=None):
    """Three recurrent steps of the kernel (from a random state) against MOAReference64, every row with an MOA (sel < K); the
    reference is pinned to the numpy oracle on the first step.  clip "median": the float32 median of the reference's influence
    at each step, so that the clamp acts on about half of the agents.  -> {check: largest error}."""
    m = steps[0][0].shape[0]
    K = len(sets)
    live = sel < K
    skip = ~live
    h0, c0 = _random_state(m, seed)
    ref = MOAReference64(sets, n, a, sel, h0, c0)
    h, c = net.state_from_rows(h0), net.state_from_rows(c0)
    errs = {}

    def note(name, err, tol):
        errs[name] = max(errs.get(name, 0.0), err)
        assert err < tol, (name, err, tol)

    tol_infl = 8 * MOA_TOL * (n - 1)
    for t, (x, joint, pl) in enumerate(steps):
        h_prev, c_prev = ref.h, ref.c
        want = ref.step(x, joint)
        bad = bad_rows(joint, a)
        assert want["pred"][live].abs().max().item() > 0.1   # not vacuous
        for div in divergences:
            ipa64, infl64 = influence64(want["pred"], want["counterfactual"], pl, joint, a, div)
            cl = clip
            if clip == "median":
                cl = float(np.float32(infl64[live & ~bad].median().item()))
                assert bool((infl64[live & ~bad] > cl).any())
                infl64 = infl64.clamp(-cl, cl)
            if a > 1:
                assert infl64[live & ~bad].abs().max().item() > 1e-3   # not vacuous
            if t == 0:
                rows = _pin_rows(edge, m, extra=np.flatnonzero(bad.cpu().numpy()), seed=seed)
                assert len(rows) <= 4096
                ref.pin(x, joint, pl, h_prev, c_prev, dict(want, influence_per_agent=ipa64, influence=infl64), rows, div, cl)
            s = raw_step(net, x, ids, joint, pl, h, c, div, cl, True)
            got = {"pred": s.pred, "counterfactual": s.counterfactual, "h": net.state_rows(s.h, m), "c": net.state_rows(s.c, m)}
            for name in ("pred", "counterfactual", "h", "c"):
                note(name, _live_err(got[name], want[name], live), MOA_TOL)
            if bool(skip.any()):   # the rows of agents without an MOA keep what the caller wrote
                for name, v in list(got.items()) + [("influence", s.influence), ("influence_per_agent", s.influence_per_agent)]:
                    assert bool((v[skip] == SENTINELS[name]).all()), name
            # NaN exactly in the envs with an invalid action
            assert torch.equal(torch.isnan(s.influence)[live], bad[live])
            assert torch.equal(torch.isnan(s.influence_per_agent)[live], bad[live, None].expand(-1, n - 1))
            ok = live & ~bad
            own_ipa, own_infl = influence64(s.pred, s.counterfactual, pl, joint, a, div, cl)
            for name, g, w in (("influence_per_agent", s.influence_per_agent, own_ipa), ("influence", s.influence, own_infl)):
                note(name + " (own logits, relative)", ((g[ok].double() - w[ok]).abs() / (1 + w[ok].abs())).max().item(), OWN_TOL)
            note("influence_per_agent (end to end)", _live_err(s.influence_per_agent, ipa64, ok), tol_infl)
            note("influence (end to end)", _live_err(s.influence, infl64, ok), tol_infl)
            if a == 1:
                assert bool((s.influence[ok] == 0).all())
            if cl != math.inf:
                assert float(s.influence[ok].max()) <= cl
            if div == "jsd":
                assert float(s.influence_per_agent[ok].max()) <= math.log(2) + 1e-6
        off = raw_step(net, x, ids, joint, pl, h, c, divergences[-1], cl, False)
        for name, g, w in (("influence", off.influence, s.influence), ("influence_per_agent", off.influence_per_agent, s.influence_per_agent),
                           ("pred", off.pred, s.pred), ("h", net.state_rows(off.h, m), got["h"]), ("c", net.state_rows(off.c, m), got["c"])):
            assert torch.equal(_bits(g[live]), _bits(w[live])), ("counterfactuals off", t, name)
        h, c = s.h, s.c
    if record is not None:
        for name, e in errs.items():
            record("max error: " + name, e)
    return errs


# ---------------------------------------------------------------------------------------------------- inputs
@pytest.fixture(scope="module")
def harvest_steps():
    """Three closed-loop steps of 65 536 Harvest envs x 5 agents: (features [M, 32] of ConvToFCNet.features on the step
    kernel's observations, joint actions int8 [B, 5] sampled by policy_step of a per-agent network, its logits [M, 8])."""
    policy = _policy()
    from sequential_social_dilemma_games_b200.batched import BatchedSSDEnv, make_config
    B, N = HARVEST_ENVS, HARVEST_AGENTS
    env = BatchedSSDEnv(make_config("harvest", num_agents=N), B, seed=29)
    pnet = policy.ConvToFCNet([policy.random_weights(num_outputs=8, seed=310 + k) for k in range(N)])
    pnet.seed_sampling(11)
    obs = env.reset()
    h, c = pnet.initial_state(B * N)
    out = []
    for _ in range(3):
        x = pnet.features(obs)
        st = pnet.policy_step(obs, h, c, features=x)
        out.append((x.clone(), st.actions.view(B, N).to(torch.int8).contiguous(), st.logits.clone()))
        h, c = st.h, st.c
        obs, _ = env.step(st.actions.view(B, N))
    torch.cuda.synchronize()
    env.close()
    pnet.close()
    assert len(torch.unique(out[-1][1])) == 8
    return out


def _int8_steps(steps):
    return [(x, j.to(torch.int8).contiguous(), pl) for x, j, pl in steps]


# ---------------------------------------------------------------------------------------------------- shared, per-agent
def test_shared_matches_float64_at_scale(harvest_steps, record_property):
    """Shared weights on 65 536 closed-loop Harvest envs x 5 agents (every CTA runs ~17 groups), KL and JSD."""
    n, a = HARVEST_AGENTS, 8
    m = HARVEST_ENVS * n
    assert _cdiv(m, GA) >= 4 * _sms()
    sets = [_weights(n, a, seed=1100)]
    net = _policy().MOANet(sets[0], n)
    sel = torch.zeros(m, dtype=torch.long, device="cuda")
    check_at_scale(net, sets, n, a, harvest_steps, sel, shared_edges(m), divergences=("kl", "jsd"), seed=1, record=record_property)
    net.close()


@pytest.mark.parametrize("source,n,a,tail,divergence,clip", [
    pytest.param("harvest", 5, 8, None, "kl", math.inf, id="harvest-5-8"),
    pytest.param("random", 5, 9, 77, "jsd", math.inf, id="random-5-9"),
    pytest.param("random", 16, 4, 5, "kl", "median", id="random-16-4-clip"),
])
def test_per_agent_matches_float64_at_scale(source, n, a, tail, divergence, clip, request, record_property):
    """Per-agent weights: the Harvest inputs (B = 65 536), or B = 4 floor(sms / N) 128 + tail random envs (N floor(sms / N) CTAs,
    one weight set each)."""
    sms = _sms()
    steps = request.getfixturevalue("harvest_steps") if source == "harvest" else \
        _int8_steps(_inputs(4 * (sms // n) * GA + tail, n, a, seed=1200 + n))
    B = steps[0][1].shape[0]
    assert _cdiv(B, GA) >= 4 * (sms // n)   # every CTA of a weight set runs at least four groups
    sets = [_weights(n, a, seed=1300 + 20 * n + k) for k in range(n)]
    net = _policy().MOANet(sets, n)
    sel = torch.arange(B * n, device="cuda") % n
    check_at_scale(net, sets, n, a, steps, sel, per_agent_edges(B, n), divergences=(divergence,), clip=clip, seed=n,
                   record=record_property)
    net.close()


# ---------------------------------------------------------------------------------------------------- pool
def _pool_ctas(m, K):
    """The pool's grid: min(max_tiles(M, K), #SMs) CTAs (ssd_policy.h)."""
    return min(_cdiv(m, GA) + K, _sms())


def _tile_sets_per_cta(counts, ctas):
    """Weight sets each CTA touches: the tiles are in set order, ceil(count / 128) per set, CTA c takes [c T / G, (c + 1) T / G)."""
    tiles = np.repeat(np.arange(len(counts)), (np.asarray(counts) + GA - 1) // GA)
    nt = len(tiles)
    return nt, [len(set(tiles[c * nt // ctas:(c + 1) * nt // ctas].tolist())) for c in range(ctas)]


def _pool_ids_k40(m, seed):
    """~1 % of the agents skipped (ids 40..255); sets 0, 1 and 2 hold 1, 127 and 129 agents (a lone row, a partial tile, a
    full tile and a row), the other sets share the rest at random."""
    rng = np.random.RandomState(seed)
    K = 40
    skipped = m // 100
    fixed = np.concatenate([[0], np.full(127, 1), np.full(129, 2), rng.randint(K, 256, skipped)])
    ids = np.concatenate([fixed, rng.randint(3, K, m - len(fixed))])
    rng.shuffle(ids)
    return ids


def _pool_ids_k255(seed):
    """Set k holds 129 + 37 k mod 256 agents (2 or 3 tiles, the last partial); ~1 % of the agents skipped (id 255), enough
    to make M a multiple of 5."""
    K = 255
    counts = 129 + (37 * np.arange(K)) % 256
    pad = (-int(counts.sum())) % 5 + 5 * 130
    ids = np.concatenate([np.repeat(np.arange(K), counts), np.full(pad, 255)])
    np.random.RandomState(seed).shuffle(ids)
    return ids


@pytest.mark.parametrize("K", [40, 255])
def test_pool_matches_float64_at_scale(K, harvest_steps, record_property):
    """K = 40 on the 65 536 x 5 Harvest inputs with ~1 % skipped agents (KL); K = 255 on random inputs (JSD, clipped), sized so
    that every CTA runs at least four tiles and crosses at least one weight-set boundary (K - 1 boundaries over #SMs CTAs).
    The pin covers every agent of the small sets (sets 0-2 of K = 40, three sets spread over K = 255)."""
    n, a = 5, 8
    if K == 40:
        steps = harvest_steps
        m = steps[0][0].shape[0]
        ids_np = _pool_ids_k40(m, seed=40)
        small = np.flatnonzero(ids_np < 3)
        div, clip = "kl", math.inf
    else:
        ids_np = _pool_ids_k255(seed=255)
        m = len(ids_np)
        steps = _int8_steps(_inputs(m // n, n, a, seed=1400))
        small = np.flatnonzero(np.isin(ids_np, [0, 127, 254]))
        div, clip = "jsd", "median"
    counts = np.bincount(ids_np, minlength=256)[:K]
    assert 0.005 < (ids_np >= K).mean() < 0.02
    ctas = _pool_ctas(m, K)
    nt, sets_per_cta = _tile_sets_per_cta(counts, ctas)
    assert ctas == _sms() and nt >= 4 * ctas   # every CTA runs at least four tiles
    if K == 255:
        assert min(sets_per_cta) >= 2   # every CTA reloads the resident weights at least once
    sets = [_weights(n, a, seed=1500 + k) for k in range(K)]
    pool = _policy().MOAPool(sets, n)
    ids = torch.from_numpy(ids_np.astype(np.uint8)).cuda()
    sel = ids.long()
    edge = np.concatenate([small] + [np.flatnonzero(ids_np == k)[[0, -1]] for k in range(0, K, max(1, K // 32)) if counts[k]])
    check_at_scale(pool, sets, n, a, steps, sel, edge, ids=ids, divergences=(div,), clip=clip, seed=K, record=record_property)
    pool.close()


# ---------------------------------------------------------------------------------------------------- invalid actions
def _invalid_envs(B, n_groups, env_of_group, seed):
    """~0.1 % of the envs plus the envs at group boundaries (the env where one of 16 groups spread over the batch starts and
    the env before it) and the last env (the ragged tail)."""
    rng = np.random.RandomState(seed)
    starts = env_of_group(np.unique(np.linspace(1, n_groups - 1, 16).astype(np.int64)))
    envs = np.concatenate([rng.choice(B, max(1, B // 1000), replace=False), starts, starts - 1, [B - 1]])
    return np.unique(envs)


@pytest.mark.parametrize("kind,a", [("shared", 8), ("per_agent", 9)])
def test_invalid_actions_at_scale(kind, a, record_property):
    """One action of ~0.1 % of the envs is -1, A, 127 or -128 (through the C ABI, unclamped), in envs at group boundaries
    and in the ragged tail too: the influence is NaN exactly in those envs, every other output matches the reference (a zero
    one-hot row).  A = 8 runs the extra drain of an invalid own action on warps 0-3, A = 9 on warps 4-7."""
    n, sms = 5, _sms()
    if kind == "shared":
        B = _cdiv(4 * sms * GA + 77, n)
        n_groups = _cdiv(B * n, GA)
        assert n_groups >= 4 * sms
        env_of_group = lambda g: (g * GA) // n   # group g starts at agent 128 g
        edge = shared_edges(B * n)
    else:
        B = 4 * (sms // n) * GA + 77
        n_groups = _cdiv(B, GA)
        assert n_groups >= 4 * (sms // n)
        env_of_group = lambda g: g * GA          # group g of every weight set starts at env 128 g
        edge = per_agent_edges(B, n)
    envs = _invalid_envs(B, n_groups, env_of_group, seed=a)
    assert B - 1 in envs and 0.001 * B <= len(envs) < 0.01 * B
    rng = np.random.RandomState(a)
    steps = []
    for t, (x, joint, pl) in enumerate(_int8_steps(_inputs(B, n, a, seed=1600 + a))):
        j = joint.clone()
        vals = np.array([-1, a, 127, -128])[(np.arange(len(envs)) + t) % 4]
        j[torch.from_numpy(envs).cuda(), torch.from_numpy(rng.randint(0, n, len(envs))).cuda()] = torch.from_numpy(vals.astype(np.int8)).cuda()
        steps.append((x, j.contiguous(), pl))
    sets = [_weights(n, a, seed=1700 + k) for k in range(1 if kind == "shared" else n)]
    net = _policy().MOANet(sets[0] if kind == "shared" else sets, n)
    sel = torch.zeros(B * n, dtype=torch.long, device="cuda") if kind == "shared" else torch.arange(B * n, device="cuda") % n
    check_at_scale(net, sets, n, a, steps, sel, edge, seed=a, record=record_property)
    net.close()
