"""Times the per-agent policy network (one weight set per agent id, ConvToFCNet([w_0, ..., w_4])) against the shared one on
the observations of the headline workload: 65 536 Harvest envs x 5 agents = 327 680 agents per call.  First checks that P
copies of one weight set give exactly the shared network's features, logits, value, state and actions at that size; then
alternates the two networks over several rounds on the same observations and prints trunk, head (ssd_policy_lstm_heads
alone), forward and closed-loop (env.step -> act) times of both, and the per-step cost of running per-agent weights without
the per-agent kernels: gather obs[:, n] into a contiguous copy, run network n on it, scatter its actions into [B, N].
Run on the GPU box: python profiles/policy_per_agent_bench.py [num_envs] [rounds]"""
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


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 7
    N, A = 5, 8
    print("card: %s" % card())
    env = BatchedSSDEnv(make_config("harvest", num_agents=N), B, seed=0)
    obs = env.reset()
    acts = torch.randint(0, A, (B, N), dtype=torch.int8, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
    for _ in range(20):
        obs, _ = env.step(acts)
    obs = obs.clone()
    M = B * N

    # ---- identical weights: the per-agent kernels reproduce the shared ones at this size, bitwise
    w = policy.random_weights(num_outputs=A, seed=0)
    shared, same = policy.ConvToFCNet(w), policy.ConvToFCNet([w] * N)
    hs, cs = shared.initial_state(M)
    hq, cq = same.initial_state(M)
    assert torch.equal(shared.features(obs), same.features(obs)), "features differ"
    for k in range(2):
        ls, vs, hs2, cs2 = shared.forward(obs, hs, cs)
        lq, vq, hq2, cq2 = same.forward(obs, hq, cq)
        assert torch.equal(ls, lq) and torch.equal(vs, vq), "logits / value differ"
        assert torch.equal(shared.state_rows(hs2, M), same.state_rows(hq2, M)), "h differs"
        assert torch.equal(shared.state_rows(cs2, M), same.state_rows(cq2, M)), "c differs"
        shared.seed_sampling(7 + k)
        same.seed_sampling(7 + k)
        a_s, _, hs, cs = shared.act(obs, hs, cs)
        a_q, _, hq, cq = same.act(obs, hq, cq)
        assert torch.equal(a_s, a_q), "actions differ"
    print("identical weights x %d == shared network at %d agents: features, logits, value, h, c, actions bitwise (2 steps)" % (N, M))
    same.close()

    # ---- distinct weights: the reference's per-agent configuration
    ws = [policy.random_weights(num_outputs=A, seed=10 + n) for n in range(N)]
    per = policy.ConvToFCNet(ws)
    singles = [policy.ConvToFCNet(x) for x in ws]   # the workaround: one shared-weights network per agent id
    nets = {"shared": shared, "per_agent": per}
    feats = {k: torch.empty((M, 32), device="cuda") for k in nets}
    state = {k: list(n.initial_state(M)) for k, n in nets.items()}
    out = {k: (torch.empty_like(state[k][0]), torch.empty_like(state[k][1]), torch.empty((M, A), device="cuda"),
               torch.empty((M,), device="cuda"), torch.empty((M,), dtype=torch.int8, device="cuda")) for k in nets}
    p = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for k, n in nets.items():
        n.features(obs, out=feats[k])

    def trunk(k):
        return lambda: nets[k].features(obs, out=feats[k])

    def head(k):
        h, c = state[k]
        hn, cn, lg, vl, ac = out[k]
        return lambda: _lib.check(_lib.lib.ssd_policy_lstm_heads(nets[k]._h, p(feats[k]), p(h), p(c), p(hn), p(cn), p(lg), p(vl), p(ac), M, 1, 2, st))

    def forward(k):
        return lambda: nets[k].forward(obs, *state[k])

    loop_state = {k: {"obs": obs.clone(), "h": state[k][0].clone(), "c": state[k][1].clone()} for k in nets}

    def loop(k):
        s = loop_state[k]

        def f():
            a, _, s["h"], s["c"] = nets[k].act(s["obs"], s["h"], s["c"])
            s["obs"], _ = env.step(a.view(B, N))
        return f

    ws_state = [list(n.initial_state(B)) for n in singles]
    ws_obs = {"obs": obs.clone()}
    a_full = torch.empty((B, N), dtype=torch.int8, device="cuda")

    def workaround():   # gather obs[:, n], N trunk + N head launches, scatter the actions, env.step
        o = ws_obs["obs"]
        for n, net in enumerate(singles):
            a, _, ws_state[n][0], ws_state[n][1] = net.act(o[:, n].contiguous(), ws_state[n][0], ws_state[n][1])
            a_full[:, n] = a
        ws_obs["obs"], _ = env.step(a_full)

    def workaround_policy_only():   # the same without env.step, on fixed observations
        for n, net in enumerate(singles):
            a, _, ws_state[n][0], ws_state[n][1] = net.act(obs[:, n].contiguous(), ws_state[n][0], ws_state[n][1])
            a_full[:, n] = a

    cases = [("trunk", trunk, 50), ("head", head, 50), ("forward", forward, 20), ("closed_loop", loop, 20)]
    res = {(c, k): [] for c, _, _ in cases for k in nets}
    res_wa, res_wa_pol = [], []
    for r in range(rounds):   # alternate: shared, per-agent, shared, ... on the same observations
        for c, mk, iters in cases:
            for k in nets:
                res[(c, k)].append(timed(mk(k), iters))
        res_wa.append(timed(workaround, 20))
        res_wa_pol.append(timed(workaround_policy_only, 20))
    print("%d envs x %d agents = %d agents; %d alternating rounds; median [min, max] ms per call" % (B, N, M, rounds))
    for c, _, _ in cases:
        med = {k: float(np.median(res[(c, k)])) for k in nets}
        print("  %-12s shared %.4f [%.4f, %.4f]   per_agent %.4f [%.4f, %.4f]   per_agent / shared %.3f" % (
            c, med["shared"], min(res[(c, "shared")]), max(res[(c, "shared")]),
            med["per_agent"], min(res[(c, "per_agent")]), max(res[(c, "per_agent")]), med["per_agent"] / med["shared"]))
    print("  workaround (gather obs[:, n] + %d x (trunk + head) + scatter), policy only: %.4f [%.4f, %.4f] ms per step" % (
        N, float(np.median(res_wa_pol)), min(res_wa_pol), max(res_wa_pol)))
    print("  workaround closed loop (+ env.step): %.4f [%.4f, %.4f] ms per step" % (float(np.median(res_wa)), min(res_wa), max(res_wa)))
    env.close()


if __name__ == "__main__":
    main()
