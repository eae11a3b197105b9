"""Times MOAPool.step (ssd_moa_pool_step: K MOA weight sets, agent m evaluated with set policy_ids[m]) against what a caller runs
without it, on the trunk features of 65 536 Harvest envs x 5 agents = 327 680 agents per call (A = 8), with the policy's own
sampled actions and logits of the step kernel's observations:
  (a) 1 set                                   MOAPool.step vs MOANet shared
  (b) 5 sets, ids[b, n] = n                   MOAPool.step vs MOANet per agent
  (c) 40 sets: 8 seeds x 5, env b -> seed b mod 8, ids[b, n] = 5 (b mod 8) + n
                                              MOAPool.step vs the per-seed workaround: per seed, gather its envs' features,
                                              joint actions and logits, run that seed's per-agent MOANet, scatter pred,
                                              influence_per_agent and influence back (each seed's state kept in its own MOANet's
                                              layout, so no state copies: the cheapest form of the workaround)
  (d) 40 sets, random ids (random teams)      MOAPool.step vs the row-wise workaround: 40 shared MOANets on all agents, rows
                                              selected by id
  closed loop of (c): env.step + PolicyPool.features + PolicyPool.policy_step + MOAPool.step per step, with policy_step given
  the features (one trunk call per step) and without (the trunk runs again inside policy_step).
Every configuration is first checked against its reference at this size (bitwise: pred, influence, influence_per_agent, h', c').
Then alternating rounds, median [min, max] ms per call (CUDA events around `iters` back-to-back calls); the card's name, power
limit and max SM clock are read in the same run.  Run on a GPU: python profiles/moa_pool_bench.py [num_envs] [rounds]"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, HERE)
from moa_bench import card, timed  # noqa: E402
from sequential_social_dilemma_games_b200 import policy  # noqa: E402
from sequential_social_dilemma_games_b200.batched import BatchedSSDEnv, make_config  # noqa: E402

N, A, SEEDS = 5, 8, 8


def rows(net, s, m):
    return [s.pred, s.influence, s.influence_per_agent, net.state_rows(s.h, m), net.state_rows(s.c, m)]


def same(got, want, what):
    for name, g, w in zip(("pred", "influence", "influence_per_agent", "h", "c"), got, want):
        assert torch.equal(g, w), "%s: %s differs from the reference" % (what, name)
    print("%s: equal to the reference, bitwise" % what)


class PerSeed(object):
    """The per-seed workaround of (c): seed s owns envs b = s mod SEEDS and a per-agent MOANet."""

    def __init__(self, sets, B, h_rows, c_rows):
        self.nets = [policy.MOANet(sets[N * s:N * (s + 1)], N) for s in range(SEEDS)]
        self.envs = [torch.arange(s, B, SEEDS, device="cuda") for s in range(SEEDS)]
        self.agents = [(e[:, None] * N + torch.arange(N, device="cuda")[None, :]).reshape(-1) for e in self.envs]
        self.state = [(net.state_from_rows(h_rows[a]), net.state_from_rows(c_rows[a])) for net, a in zip(self.nets, self.agents)]

    def step(self, x, joint, pl, out):
        pred, infl, ipa = out
        res = []
        for net, e, a, (h, c) in zip(self.nets, self.envs, self.agents, self.state):
            s = net.step(x[a], joint[e], pl[a], h, c)
            pred[a], infl[a], ipa[a] = s.pred, s.influence, s.influence_per_agent
            res.append(s)
        return res


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    M = B * N
    print(card())
    print("%d Harvest envs x %d agents = %d agents per call, A = %d, %d alternating rounds" % (B, N, M, A, rounds))
    env = BatchedSSDEnv(make_config("harvest", num_agents=N), B, seed=1)
    obs = env.reset()
    pnet = policy.ConvToFCNet(policy.random_weights(num_outputs=A, seed=0))
    x = pnet.features(obs)
    h0, c0 = pnet.initial_state(M)
    st = pnet.policy_step(obs, h0, c0)
    joint, pl = st.actions.view(B, N), st.logits
    pnet.close()
    g = torch.Generator(device="cuda").manual_seed(2)
    h_rows = 0.5 * torch.randn((M, 128), device="cuda", generator=g)
    c_rows = 0.5 * torch.randn((M, 128), device="cuda", generator=g)
    sets = [policy.random_moa_weights(N, A, seed=10 + k) for k in range(SEEDS * N)]
    b_idx, n_idx = torch.arange(B, device="cuda")[:, None], torch.arange(N, device="cuda")[None, :]
    results = []

    def run(label, variants, iters):
        times = {k: [] for k in variants}
        for _ in range(rounds):
            for k, fn in variants.items():
                times[k].append(timed(fn, iters[k]))
        print(label)
        med = {}
        for k, ts in times.items():
            ts = sorted(ts)
            med[k] = ts[len(ts) // 2]
            print("  %-28s median %8.3f ms [%.3f, %.3f]" % (k, med[k], ts[0], ts[-1]))
        results.append((label, med))
        return med

    # (a) one set, (b) five sets with ids = n
    for label, ws, ids in (("(a) 1 set", sets[:1], torch.zeros((B, N), dtype=torch.uint8, device="cuda")),
                           ("(b) 5 sets, ids = n", sets[:N], n_idx.expand(B, N).to(torch.uint8).contiguous())):
        net = policy.MOANet(ws if len(ws) > 1 else ws[0], N)
        pool = policy.MOAPool(ws, N)
        hn, cn = net.state_from_rows(h_rows), net.state_from_rows(c_rows)
        hp, cp = pool.state_from_rows(h_rows), pool.state_from_rows(c_rows)
        same(rows(pool, pool.step(x, ids, joint, pl, hp, cp), M), rows(net, net.step(x, joint, pl, hn, cn), M), label)
        run(label, {"MOAPool.step": lambda: pool.step(x, ids, joint, pl, hp, cp),
                    "MOANet.step": lambda: net.step(x, joint, pl, hn, cn)}, {"MOAPool.step": 20, "MOANet.step": 20})
        net.close()
        pool.close()
        torch.cuda.empty_cache()

    # (c) 8 seeds x 5 agents, env b -> seed b mod 8
    ids_c = (N * (b_idx % SEEDS) + n_idx).to(torch.uint8)
    pool = policy.MOAPool(sets, N)
    hp, cp = pool.state_from_rows(h_rows), pool.state_from_rows(c_rows)
    ws = PerSeed(sets, B, h_rows, c_rows)
    out = [torch.empty((M, N - 1, A), device="cuda"), torch.empty((M,), device="cuda"), torch.empty((M, N - 1), device="cuda")]
    s = pool.step(x, ids_c, joint, pl, hp, cp)
    per = ws.step(x, joint, pl, out)
    hw, cw = torch.empty((M, 128), device="cuda"), torch.empty((M, 128), device="cuda")
    for net, a, r in zip(ws.nets, ws.agents, per):
        hw[a], cw[a] = net.state_rows(r.h, a.numel()), net.state_rows(r.c, a.numel())
    same(rows(pool, s, M), out + [hw, cw], "(c) 8 seeds x 5")
    run("(c) 40 sets, 8 seeds x 5, env b -> seed b mod 8", {"MOAPool.step": lambda: pool.step(x, ids_c, joint, pl, hp, cp),
                                                            "per-seed gather/scatter": lambda: ws.step(x, joint, pl, out)},
        {"MOAPool.step": 20, "per-seed gather/scatter": 10})
    del ws, per

    # (d) random teams
    ids_d = torch.randint(0, SEEDS * N, (B, N), dtype=torch.uint8, device="cuda", generator=g)
    refs = [policy.MOANet(w, N) for w in sets]
    hs, cs = refs[0].state_from_rows(h_rows), refs[0].state_from_rows(c_rows)   # a shared MOA's layout = the pool's
    flat = ids_d.reshape(-1).long()

    def rowwise(with_state=False):   # 40 MOA calls, rows selected by id (and, for the check, the state rows)
        res = [torch.empty((M, N - 1, A), device="cuda"), torch.empty((M,), device="cuda"), torch.empty((M, N - 1), device="cuda")]
        if with_state:
            res += [torch.empty((M, 128), device="cuda"), torch.empty((M, 128), device="cuda")]
        for k, net in enumerate(refs):
            r = net.step(x, joint, pl, hs, cs)
            sel = flat == k
            outs = (r.pred, r.influence, r.influence_per_agent) + ((net.state_rows(r.h, M), net.state_rows(r.c, M)) if with_state else ())
            for o, t in zip(res, outs):
                o[sel] = t[sel]
        return res

    s = pool.step(x, ids_d, joint, pl, hp, cp)
    same(rows(pool, s, M), rowwise(with_state=True), "(d) 40 sets, random teams")

    run("(d) 40 sets, random teams", {"MOAPool.step": lambda: pool.step(x, ids_d, joint, pl, hp, cp), "40 MOANet calls + select": rowwise},
        {"MOAPool.step": 20, "40 MOANet calls + select": 2})
    for net in refs:
        net.close()
    del refs
    torch.cuda.empty_cache()

    # closed loop of (c)
    ppool = policy.PolicyPool([policy.random_weights(num_outputs=A, seed=100 + k) for k in range(SEEDS * N)])
    ppool.seed_sampling(3)
    h, c = ppool.initial_state(M)
    hm, cm = pool.initial_state(M)
    state = {"obs": obs}

    def loop(features):
        o = state["obs"]
        xf = ppool.features(o, ids_c)
        stp = ppool.policy_step(o, ids_c, h, c, features=xf) if features else ppool.policy_step(o, ids_c, h, c)
        pool.step(xf, ids_c, stp.actions.view(B, N), stp.logits, hm, cm)
        state["obs"], _ = env.step(stp.actions.view(B, N))

    xf = ppool.features(obs, ids_c)
    a1 = ppool.policy_step(obs, ids_c, h, c, mode="greedy", features=xf)
    a2 = ppool.policy_step(obs, ids_c, h, c, mode="greedy")
    assert torch.equal(a1.logits, a2.logits) and torch.equal(a1.actions, a2.actions)
    print("closed loop: policy_step with features equals policy_step without, bitwise")
    run("closed loop (c): env.step + trunk + policy_step + MOAPool.step", {"features=x": lambda: loop(True), "trunk twice": lambda: loop(False)},
        {"features=x": 10, "trunk twice": 10})
    env.close()
    ppool.close()
    pool.close()

    print("\nsummary (median ms per call):")
    for label, med in results:
        print("  %-62s %s" % (label, ", ".join("%s %.3f" % kv for kv in med.items())))


if __name__ == "__main__":
    main()
