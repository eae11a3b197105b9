"""Times the policy pool (PolicyPool: K weight sets, a uint8 policy id per agent and call) on the observations of the headline
workload, 65 536 Harvest envs x 5 agents = 327 680 agents per call, against the network each configuration replaces:
  (a) a pool of 1, every id 0                          vs the shared network ConvToFCNet(w)
  (b) a pool of 5, ids[b, n] = n                       vs the per-agent network ConvToFCNet([w_0..w_4])
  (c) 40 sets = 8 seeds x 5 agents, ids[b, n] = 5 (b mod 8) + n          vs the per-policy gather-and-loop workaround
  (d) 40 sets, a random team per env: ids[b, n] = 5 s_b,n + n, s random  vs the same workaround
Each configuration is first checked bitwise against its reference at this size (features, logits, value, h, c, actions).
Then the configurations are timed in alternating rounds on the same observations (median ms per call): trunk, head
(ssd_policy_pool_lstm_heads alone, its assignment included), forward, closed loop (env.step -> act).  A separate
torch.profiler pass gives the device time per call of the assignment kernels (count + plan + scatter) and of the pool
trunk and head kernels, and the script counts the weight reloads (policy switches inside the CTAs' tile ranges).
The workaround keeps agent-major state rows [M, 128] and, per policy, gathers obs / h / c rows, runs a shared network,
scatters actions and state back.
Run on the GPU box: python profiles/policy_pool_bench.py [num_envs] [rounds] [out_dir]"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from sequential_social_dilemma_games_b200 import _lib, policy  # noqa: E402
from sequential_social_dilemma_games_b200.batched import BatchedSSDEnv, make_config  # noqa: E402


def timed(fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "power limit not readable (%s)" % e
    return "%s, %s" % (name, q)


def switches(ids, K, sms):
    """Weight reloads of the pool kernels: policy changes inside the CTAs' contiguous tile ranges (host model of the plan)."""
    counts = np.bincount(ids.reshape(-1).cpu().numpy().astype(np.int64), minlength=256)[:K]
    tiles = np.concatenate([np.full((c + 127) // 128, k) for k, c in enumerate(counts)])
    T = len(tiles)
    G = min(sms, (ids.numel() + 127) // 128 + K)
    n = 0
    for c in range(G):
        r = tiles[T * c // G:T * (c + 1) // G]
        n += int(np.count_nonzero(r[1:] != r[:-1]))
    return n, T, G


class Workaround(object):
    """Per-policy gather-and-loop with a shared network per weight set and agent-major state rows."""

    def __init__(self, sets, ids):
        self.nets = [policy.ConvToFCNet(w) for w in sets]
        flat = ids.reshape(-1).long()
        self.idx = [torch.nonzero(flat == k).squeeze(1) for k in range(len(sets))]   # fixed for the episode
        self.idx = [(k, i) for k, i in enumerate(self.idx) if i.numel()]
        M = flat.numel()
        self.h = torch.zeros((M, 128), device="cuda")
        self.c = torch.zeros((M, 128), device="cuda")
        self.a = torch.empty((M,), dtype=torch.int8, device="cuda")

    def act(self, obs):
        flat = obs.reshape(-1, 15, 15, 3)
        for k, i in self.idx:
            net = self.nets[k]
            m = i.numel()
            a, _, h, c = net.act(flat[i], net.state_from_rows(self.h[i]), net.state_from_rows(self.c[i]))
            self.a[i] = a
            self.h[i] = net.state_rows(h, m)
            self.c[i] = net.state_rows(c, m)
        return self.a


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    out_dir = sys.argv[3] if len(sys.argv) > 3 else None
    N, A, S = 5, 8, 8
    M = B * N
    print("card: %s" % card())
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    env = BatchedSSDEnv(make_config("harvest", num_agents=N), B, seed=0)
    obs = env.reset()
    acts = torch.randint(0, A, (B, N), dtype=torch.int8, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
    for _ in range(20):
        obs, _ = env.step(acts)
    obs = obs.clone()
    flat = obs.reshape(M, 15, 15, 3)

    w1 = [policy.random_weights(num_outputs=A, seed=0)]
    w5 = [policy.random_weights(num_outputs=A, seed=10 + n) for n in range(N)]
    w40 = [policy.random_weights(num_outputs=A, seed=100 + k) for k in range(S * N)]
    slot = torch.arange(N, device="cuda")[None, :]
    env_b = torch.arange(B, device="cuda")[:, None]
    team = torch.randint(0, S, (B, N), device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    ids = {"a": torch.zeros((B, N), dtype=torch.uint8, device="cuda"),
           "b": slot.expand(B, N).to(torch.uint8).contiguous(),
           "c": (N * (env_b % S) + slot).to(torch.uint8),
           "d": (N * team + slot).to(torch.uint8)}
    pools = {"a": policy.PolicyPool(w1), "b": policy.PolicyPool(w5), "c": policy.PolicyPool(w40)}
    pools["d"] = pools["c"]
    base = {"a": policy.ConvToFCNet(w1[0]), "b": policy.ConvToFCNet(w5)}

    # ---- bitwise checks at this size: (a), (b) against their networks; (c), (d) against the row-wise reference
    for k in "ab":
        p, n = pools[k], base[k]
        hp, cp = p.initial_state(M)
        hn, cn = n.initial_state(M)
        assert torch.equal(p.features(obs, ids[k]), n.features(obs)), k
        for t in range(2):
            lp, vp, hp2, cp2 = p.forward(obs, ids[k], hp, cp)
            ln, vn, hn2, cn2 = n.forward(obs, hn, cn)
            assert torch.equal(lp, ln) and torch.equal(vp, vn), k
            assert torch.equal(p.state_rows(hp2, M), n.state_rows(hn2, M)) and torch.equal(p.state_rows(cp2, M), n.state_rows(cn2, M)), k
            p.seed_sampling(7 + t)
            n.seed_sampling(7 + t)
            ap, _, hp, cp = p.act(obs, ids[k], hp, cp)
            an, _, hn, cn = n.act(obs, hn, cn)
            assert torch.equal(ap, an), k
    ref = [policy.ConvToFCNet(w) for w in w40]
    for k in "cd":
        p = pools[k]
        sel = ids[k].reshape(-1).long()
        h, c = p.initial_state(M)
        p.seed_sampling(3)
        f = p.features(obs, ids[k])
        lg, v, h2, c2 = p.forward(obs, ids[k], h, c)
        a, _, _, _ = p.act(obs, ids[k], h, c)
        rows_h, rows_c = p.state_rows(h2, M), p.state_rows(c2, M)
        for q, net in enumerate(ref):
            m = sel == q
            net.seed_sampling(3)
            assert torch.equal(f[m], net.features(obs)[m]), (k, q)
            l1, v1, h1, c1 = net.forward(obs, h, c)
            a1, _, _, _ = net.act(obs, h, c)
            assert torch.equal(lg[m], l1[m]) and torch.equal(v[m], v1[m]) and torch.equal(a[m], a1[m]), (k, q)
            assert torch.equal(rows_h[m], net.state_rows(h1, M)[m]) and torch.equal(rows_c[m], net.state_rows(c1, M)[m]), (k, q)
    for r in ref:
        r.close()
    print("bitwise at %d agents: (a) == shared, (b) == per-agent, (c), (d) == row-wise reference (features, logits, value, h, c, actions)" % M)
    for k in "abcd":
        n, T, G = switches(ids[k], pools[k].num_policies, sms)
        print("  (%s) %d tiles over %d CTAs, %d weight reloads inside the CTAs' ranges" % (k, T, G, n))

    # ---- timing: every contender in alternating rounds
    p_ = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    nets = {"shared": (base["a"], None), "per_agent": (base["b"], None)}
    for k in "abcd":
        nets["pool_" + k] = (pools[k], ids[k])
    feats = {k: torch.empty((M, 32), device="cuda") for k in nets}
    state = {k: list(n.initial_state(M)) for k, (n, _) in nets.items()}
    out = {k: (torch.empty_like(state[k][0]), torch.empty_like(state[k][1]), torch.empty((M, A), device="cuda"),
               torch.empty((M,), device="cuda"), torch.empty((M,), dtype=torch.int8, device="cuda")) for k in nets}
    for k, (n, i) in nets.items():
        n.features(obs, out=feats[k]) if i is None else n.features(obs, i, out=feats[k])

    def trunk(k):
        n, i = nets[k]
        return (lambda: n.features(obs, out=feats[k])) if i is None else (lambda: n.features(obs, i, out=feats[k]))

    def head(k):
        n, i = nets[k]
        h, c = state[k]
        hn, cn, lg, vl, ac = out[k]
        if i is None:
            return lambda: _lib.check(_lib.lib.ssd_policy_lstm_heads(n._h, p_(feats[k]), p_(h), p_(c), p_(hn), p_(cn), p_(lg), p_(vl), p_(ac), M, 1, 2, st))
        return lambda: _lib.check(_lib.lib.ssd_policy_pool_lstm_heads(n._h, p_(feats[k]), p_(i), p_(h), p_(c), p_(hn), p_(cn), p_(lg), p_(vl), p_(ac),
                                                                      M, 1, 2, st))

    def forward(k):
        n, i = nets[k]
        return (lambda: n.forward(obs, *state[k])) if i is None else (lambda: n.forward(obs, i, *state[k]))

    loop_state = {k: {"obs": obs.clone(), "h": state[k][0].clone(), "c": state[k][1].clone()} for k in nets}

    def loop(k):
        n, i = nets[k]
        s = loop_state[k]

        def f():
            if i is None:
                a, _, s["h"], s["c"] = n.act(s["obs"], s["h"], s["c"])
            else:
                a, _, s["h"], s["c"] = n.act(s["obs"], i, s["h"], s["c"])
            s["obs"], _ = env.step(a.view(B, N))
        return f

    wa = {k: Workaround(w40, ids[k]) for k in "cd"}
    wa_obs = {k: {"obs": obs.clone()} for k in "cd"}

    def wa_policy(k):
        return lambda: wa[k].act(obs)

    def wa_loop(k):
        def f():
            a = wa[k].act(wa_obs[k]["obs"])
            wa_obs[k]["obs"], _ = env.step(a.view(B, N))
        return f

    cases = [("trunk", trunk, 30), ("head", head, 30), ("forward", forward, 15), ("closed_loop", loop, 15)]
    res = {(c, k): [] for c, _, _ in cases for k in nets}
    res_wa = {(c, k): [] for c in ("policy", "closed_loop") for k in "cd"}
    for r in range(rounds):
        for c, mk, iters in cases:
            for k in nets:
                res[(c, k)].append(timed(mk(k), iters))
        for k in "cd":
            res_wa[("policy", k)].append(timed(wa_policy(k), 3, warm=1))
            res_wa[("closed_loop", k)].append(timed(wa_loop(k), 3, warm=1))
    med = lambda xs: float(np.median(xs))
    print("%d envs x %d agents = %d agents; %d alternating rounds; median [min, max] ms per call" % (B, N, M, rounds))
    for c, _, _ in cases:
        print("  %s" % c)
        for k in nets:
            xs = res[(c, k)]
            print("    %-10s %.4f [%.4f, %.4f]" % (k, med(xs), min(xs), max(xs)))
        print("    ratios: pool_a / shared %.3f, pool_b / per_agent %.3f" % (med(res[(c, "pool_a")]) / med(res[(c, "shared")]),
                                                                          med(res[(c, "pool_b")]) / med(res[(c, "per_agent")])))
    for k in "cd":
        for c in ("policy", "closed_loop"):
            xs = res_wa[(c, k)]
            print("  workaround (%s) %-11s %.4f [%.4f, %.4f]   pool %s: %.4f" % (k, c, med(xs), min(xs), max(xs),
                  "forward+sample" if c == "policy" else "closed loop", med(res[("closed_loop" if c == "closed_loop" else "forward", "pool_" + k)])))

    # ---- device time per kernel (torch.profiler, a separate pass): assignment vs trunk vs head
    from torch.profiler import ProfilerActivity, profile
    calls = 10
    kern = {}
    for k in ["shared", "per_agent", "pool_a", "pool_b", "pool_c", "pool_d"]:
        f = forward(k)
        f()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(calls):
                f()
            torch.cuda.synchronize()
        agg = {}
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            if t > 0:
                agg[e.key] = agg.get(e.key, 0.0) + t / 1000.0 / calls
        kern[k] = agg
        if out_dir:
            os.makedirs(out_dir, exist_ok=True)
            prof.export_chrome_trace(os.path.join(out_dir, "pool_%s.pt.trace.json" % k))
    print("device ms per forward call by kernel (torch.profiler, %d calls)" % calls)
    for k, agg in kern.items():
        groups = {"assign": sum(v for n, v in agg.items() if "pool_count" in n or "pool_plan" in n or "pool_scatter" in n),
                  "trunk": sum(v for n, v in agg.items() if "policy_features_kernel" in n),
                  "head": sum(v for n, v in agg.items() if "lstm_heads_kernel" in n)}
        other = sum(agg.values()) - sum(groups.values())
        print("  %-10s assign %.4f  trunk %.4f  head %.4f  other %.4f" % (k, groups["assign"], groups["trunk"], groups["head"], other))
    env.close()


if __name__ == "__main__":
    main()
