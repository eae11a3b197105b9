"""Times the policy's distribution outputs (ssd_policy_lstm_heads_dist / ssd_policy_pool_lstm_heads_dist: the action of a mode, its
log-probability and the entropy, in the fused head kernel) against the plain head they extend, on the observations of the
headline workload, 65 536 Harvest envs x 5 agents = 327 680 agents per call:
  shared   one network for all agents, ConvToFCNet(w)
  pool_c   40 sets = 8 seeds x 5 agents, ids[b, n] = 5 (b mod 8) + n, as (c) of policy_pool_bench.py
Each is first checked at this size: mode 'sample' gives the plain head's actions, logits, value, h' and c' bitwise, 'greedy'
the first argmax of the logits, 'given' leaves its actions unchanged.  Then, in alternating rounds on the same features and
state (median [min, max] ms per call, CUDA events around `iters` back-to-back calls):
  head       the plain head with sampling (ssd_policy_lstm_heads / _pool_) and the _dist entry point in each mode, logp and
             entropy written;
  policy     what a learner gets per step: policy_step (trunk + _dist head, greedy) against the torch route it replaces,
             forward (trunk + plain head) then log_softmax + argmax + gather and the entropy in torch.
The features (42 MB) and the recurrent state (2 x 168 MB in, 2 x 168 MB out) do not fit the 126 MB L2, so every call streams
the state from HBM.  A separate torch.profiler pass gives the device time of the head kernel alone per variant.
Run on the GPU box: python profiles/policy_dist_bench.py [num_envs] [rounds] [out_dir]"""
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
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm,clocks.sm,clocks.mem", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "power limit / clocks not readable (%s)" % e
    return "%s, power limit, max SM clock, SM clock, memory clock: %s" % (name, q)


MODES = (("sample", _lib.ACT_SAMPLE), ("greedy", _lib.ACT_GREEDY), ("given", _lib.ACT_GIVEN))


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 7
    out_dir = sys.argv[3] if len(sys.argv) > 3 else None
    N, A, S = 5, 8, 8
    M = B * N
    print("card: %s" % card())
    env = BatchedSSDEnv(make_config("harvest", num_agents=N), B, seed=0)
    obs = env.reset()
    acts = torch.randint(0, A, (B, N), dtype=torch.int8, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
    for _ in range(20):
        obs, _ = env.step(acts)
    obs = obs.reshape(M, 15, 15, 3).clone()
    env.close()

    slot = torch.arange(N, device="cuda")[None, :]
    env_b = torch.arange(B, device="cuda")[:, None]
    ids_c = (N * (env_b % S) + slot).to(torch.uint8).reshape(M)
    nets = {"shared": (policy.ConvToFCNet(policy.random_weights(num_outputs=A, seed=0)), None),
            "pool_c": (policy.PolicyPool([policy.random_weights(num_outputs=A, seed=100 + k) for k in range(S * N)]), ids_c)}
    p_ = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    g = torch.Generator(device="cuda").manual_seed(2)
    io = {}
    for k, (n, ids) in nets.items():
        feats = n.features(obs) if ids is None else n.features(obs, ids)
        h, c = n.initial_state(M)   # a non-zero state: one step from zero
        h, c = n.forward(obs, h, c)[2:] if ids is None else n.forward(obs, ids, h, c)[2:]
        io[k] = {"x": feats, "h": h, "c": c, "hn": torch.empty_like(h), "cn": torch.empty_like(c), "lg": torch.empty((M, A), device="cuda"),
                 "v": torch.empty((M,), device="cuda"), "a": torch.empty((M,), dtype=torch.int8, device="cuda"),
                 "given": torch.randint(0, A, (M,), dtype=torch.int8, device="cuda", generator=g),
                 "lp": torch.empty((M,), device="cuda"), "en": torch.empty((M,), device="cuda")}

    def plain(k):
        n, ids = nets[k]
        b = io[k]
        args = [p_(b[q]) for q in ("x", "h", "c", "hn", "cn", "lg", "v", "a")]
        if ids is None:
            return lambda: _lib.check(_lib.lib.ssd_policy_lstm_heads(n._h, *args, M, 1, 2, st))
        return lambda: _lib.check(_lib.lib.ssd_policy_pool_lstm_heads(n._h, args[0], p_(ids), *args[1:], M, 1, 2, st))

    def dist(k, code):
        n, ids = nets[k]
        b = io[k]
        args = [p_(b[q]) for q in ("x", "h", "c", "hn", "cn", "lg", "v")]
        a = p_(b["given"] if code == _lib.ACT_GIVEN else b["a"])
        if ids is None:
            return lambda: _lib.check(_lib.lib.ssd_policy_lstm_heads_dist(n._h, *args, code, a, p_(b["lp"]), p_(b["en"]), M, 1, 2, st))
        return lambda: _lib.check(_lib.lib.ssd_policy_pool_lstm_heads_dist(n._h, args[0], p_(ids), *args[1:], code, a, p_(b["lp"]),
                                                                           p_(b["en"]), M, 1, 2, st))

    # ---- checks at this size
    for k, (n, ids) in nets.items():
        b = io[k]
        live = torch.ones((M,), dtype=torch.bool, device="cuda") if ids is None else ids.long() < n.num_policies
        out = lambda: (n.state_rows(b["hn"], M), n.state_rows(b["cn"], M), b["lg"], b["v"], b["a"])
        plain(k)()
        ref = [t[live].clone() for t in out()]
        for name, code in MODES:
            given = b["given"].clone()
            for q in ("hn", "cn", "lg", "v", "a"):
                b[q].fill_(7)
            dist(k, code)()
            got = [t[live] for t in out()]
            for q in range(4):
                assert torch.equal(got[q], ref[q]), (k, name, q)
            if code == _lib.ACT_SAMPLE:
                assert torch.equal(got[4], ref[4]), (k, name)
            elif code == _lib.ACT_GREEDY:
                assert torch.equal(got[4].long(), got[2].argmax(dim=1)), (k, name)
            else:
                assert torch.equal(b["given"], given), (k, name)
            assert bool(torch.isfinite(b["lp"][live]).all()) and bool((b["en"][live] >= 0).all()), (k, name)
    print("checked at %d agents: 'sample' == the plain head bitwise (actions, logits, value, h', c'), 'greedy' == first argmax, "
          "'given' leaves actions unchanged" % M)

    # ---- the torch route a learner would otherwise take
    def torch_route(k):
        n, ids = nets[k]
        b = io[k]
        fwd = (lambda: n.forward(obs, b["h"], b["c"])) if ids is None else (lambda: n.forward(obs, ids_c, b["h"], b["c"]))

        def f():
            lg = fwd()[0]
            ls = torch.log_softmax(lg, dim=1)
            a = ls.argmax(dim=1)
            return a, ls.gather(1, a[:, None]).squeeze(1), -(ls.exp() * ls).sum(dim=1)
        return f

    def step(k):
        n, ids = nets[k]
        b = io[k]
        return (lambda: n.policy_step(obs, b["h"], b["c"], mode="greedy")) if ids is None else \
            (lambda: n.policy_step(obs, ids_c, b["h"], b["c"], mode="greedy"))

    # ---- timing: alternating rounds
    cases = [("head", "plain", lambda k: plain(k), 40)] + [("head", "dist_" + nm, (lambda code: lambda k: dist(k, code))(cd), 40) for nm, cd in MODES]
    cases += [("policy", "torch_route", torch_route, 15), ("policy", "policy_step", step, 15)]
    res = {(k, c[1]): [] for k in nets for c in cases}
    for r in range(rounds):
        for k in nets:
            for _, name, mk, iters in cases:
                res[(k, name)].append(timed(mk(k), iters))
    med = lambda xs: float(np.median(xs))
    print("%d envs x %d agents = %d agents, %d outputs; %d alternating rounds; median [min, max] ms per call" % (B, N, M, A, rounds))
    for k in nets:
        print("  %s" % k)
        base = med(res[(k, "plain")])
        for group, name, _, _ in cases:
            xs = res[(k, name)]
            rel = "  %+.1f %% vs plain" % (100 * (med(xs) / base - 1)) if group == "head" and name != "plain" else ""
            print("    %-7s %-12s %.4f [%.4f, %.4f]%s" % (group, name, med(xs), min(xs), max(xs), rel))
        print("    policy_step / torch_route %.3f" % (med(res[(k, "policy_step")]) / med(res[(k, "torch_route")])))

    # ---- device time of the head kernel alone (torch.profiler, a separate pass)
    from torch.profiler import ProfilerActivity, profile
    calls = 20
    print("device ms per call of lstm_heads_kernel (torch.profiler, %d calls)" % calls)
    for k in nets:
        for _, name, mk, _ in cases[:4]:
            f = mk(k)
            f()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(calls):
                    f()
                torch.cuda.synchronize()
            t = 0.0
            for e in prof.key_averages():
                if "lstm_heads_kernel" in e.key:
                    dt = getattr(e, "device_time_total", None)
                    t += (dt if dt is not None else e.cuda_time_total) / 1000.0 / calls
            print("  %-7s %-12s %.4f" % (k, name, t))
            if out_dir:
                os.makedirs(out_dir, exist_ok=True)
                prof.export_chrome_trace(os.path.join(out_dir, "dist_%s_%s.pt.trace.json" % (k, name)))
    print("card after the run: %s" % card())
    for n, _ in nets.values():
        n.close()


if __name__ == "__main__":
    main()
