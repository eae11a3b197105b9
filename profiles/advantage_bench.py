"""Times postprocess.compute_advantages / vtrace (csrc/ssd_advantages.cu) on the trajectories a sampler fills, against the torch
loop over t a user would otherwise write (a few elementwise ops per step, backwards, dones as a multiply by 1 - done):
  (a) 65 536 envs x 5 agents = 327 680 agents at T = 100 and T = 1000    one pass over time (C = 1)
  (b) 64 envs x 5 agents = 320 agents at T = 1000                        time split into chunks (C > 1)
  (c) 16 380 agents (3 276 envs x 5, about 16 384) at T = 1000         chunked
  (d) 81 920 agents at T = 1000: the smallest M of one pass, next to (c) for the per-byte rate of the two paths
Each workload runs GAE with the weighted intrinsic reward (int32 rewards), discounted returns (int32 rewards) and V-trace
(clip_rho 1, clip_pg 1; int32 rewards).  Rewards and logp are random, 3 % of env steps end an episode.
Every configuration is first checked against oracle/advantage_ref.py on sampled columns within its derived bound.  Then
alternating rounds: CUDA events around back-to-back calls, median [min, max] ms per call.  Working sets below 3 x the 126 MB L2
are rotated over enough copies of the inputs that consecutive calls read different memory.  Algorithmic bytes: each input read
once, each output written once.  The card's name, power limit and max SM clock are read in the same run.
Run on a GPU: python profiles/advantage_bench.py [rounds]"""
import math
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, HERE)
from moa_bench import card  # noqa: E402
from oracle import advantage_ref as ref  # noqa: E402
from sequential_social_dilemma_games_b200 import postprocess  # noqa: E402

PEAK = 7.7e12
L2 = 126e6
GAMMA, LAMBDA, W = 0.99, 0.95, 0.1
N = 5
WORKLOADS = [("a", 100, 327680), ("a", 1000, 327680), ("b", 1000, 320), ("c", 1000, 16380), ("d", 1000, 81920)]


def make(t_count, m, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda: torch.randn((t_count, m), generator=g, device="cuda")
    return dict(rewards=torch.randint(-1, 3, (t_count, m), generator=g, device="cuda", dtype=torch.int32), values=r(),
                dones=(torch.rand((t_count, m // N), generator=g, device="cuda") < 0.03).to(torch.uint8),
                bootstrap=torch.randn((m,), generator=g, device="cuda"), intrinsic=torch.rand((t_count, m), generator=g, device="cuda"),
                target_logp=0.3 * r() - 1.5, behaviour_logp=0.3 * r() - 1.5)


def call(mode, x):
    a = (x["rewards"], x["values"], x["dones"], x["bootstrap"])
    if mode == "gae":
        return postprocess.compute_advantages(*a, gamma=GAMMA, lambda_=LAMBDA, intrinsic=x["intrinsic"], intrinsic_weight=W)
    if mode == "returns":
        return postprocess.compute_advantages(*a, gamma=GAMMA, lambda_=LAMBDA, use_gae=False)
    return tuple(postprocess.vtrace(*a, x["target_logp"], x["behaviour_logp"], gamma=GAMMA, clip_rho_threshold=1.0,
                                    clip_pg_rho_threshold=1.0))


def torch_loop(mode, x):
    """What a user writes without the library: a loop over t, backwards, on [M] slices."""
    t_count, m = x["values"].shape
    v, boot = x["values"], x["bootstrap"]
    nd = 1.0 - x["dones"].float().repeat_interleave(N, dim=1)
    r = x["rewards"].float() + W * x["intrinsic"] if mode == "gae" else x["rewards"].float()
    out0, out1 = torch.empty_like(v), torch.empty_like(v)
    if mode == "returns":
        acc = boot
        for t in range(t_count - 1, -1, -1):
            acc = r[t] + GAMMA * nd[t] * acc
            out0[t] = acc
        return out0, None
    if mode == "gae":
        acc, vn = torch.zeros_like(boot), boot
        for t in range(t_count - 1, -1, -1):
            acc = r[t] + GAMMA * nd[t] * vn - v[t] + GAMMA * LAMBDA * nd[t] * acc
            out0[t] = acc
            vn = v[t]
        return out0, out0 + v
    rho = torch.exp(x["target_logp"] - x["behaviour_logp"])
    rb, cs = rho.clamp(max=1.0), rho.clamp(max=1.0)
    acc, vn, vsn = torch.zeros_like(boot), boot, boot
    for t in range(t_count - 1, -1, -1):
        acc = rb[t] * (r[t] + GAMMA * nd[t] * vn - v[t]) + GAMMA * cs[t] * nd[t] * acc
        out0[t] = acc + v[t]
        out1[t] = rb[t] * (r[t] + GAMMA * nd[t] * vsn - v[t])
        vn, vsn = v[t], out0[t]
    return out0, out1


def algorithmic_bytes(mode, t_count, m):
    per = {"gae": 4 + 4 + 4 + 8, "returns": 4 + 4, "vtrace": 4 + 4 + 8 + 8}[mode]   # reads then writes, per agent-step
    return t_count * m * per + t_count * (m // N) + 4 * m


def check(mode, x, out):
    m = x["values"].shape[1]
    rng = np.random.RandomState(0)
    cols = np.unique(np.concatenate([np.arange(4), rng.choice(m, min(m, 96), replace=False), [m - 1]]))
    ci = torch.as_tensor(cols, device="cuda")
    h = {k: v[..., ci].cpu().numpy() for k, v in x.items() if k != "dones"}
    d = x["dones"][:, ci // N].cpu().numpy()
    if mode == "vtrace":
        want = ref.vtrace(h["rewards"], h["values"], d, h["bootstrap"], h["target_logp"], h["behaviour_logp"], GAMMA, 1.0, 1.0)
        tol = ref.error_bound("vtrace", h["rewards"], h["values"], d, h["bootstrap"], GAMMA, 1.0, None, 0.0, h["target_logp"],
                              h["behaviour_logp"], 1.0, 1.0)
    elif mode == "gae":
        want = ref.compute_advantages(h["rewards"], h["values"], d, h["bootstrap"], GAMMA, LAMBDA, True, h["intrinsic"], W)
        tol = ref.error_bound("gae", h["rewards"], h["values"], d, h["bootstrap"], GAMMA, LAMBDA, h["intrinsic"], W)
    else:
        want = ref.compute_advantages(h["rewards"], h["values"], d, h["bootstrap"], GAMMA, LAMBDA, False)
        tol = ref.error_bound("returns", h["rewards"], h["values"], d, h["bootstrap"], GAMMA)
    worst = 0.0
    for got, w_, t_ in zip(out, want, tol):
        if w_ is None:
            continue
        err = np.abs(got[:, ci].double().cpu().numpy() - w_)
        assert (err <= t_).all(), (mode, float(err.max()))
        worst = max(worst, float(err.max()))
    return worst


def events(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def graphed(mode, x, iters):
    """ms per call of `iters` calls captured in one CUDA graph: the GPU time without the host's ctypes and checks per call."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        call(mode, x)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(iters):
            call(mode, x)
    g.replay()
    torch.cuda.synchronize()
    return events(lambda i: g.replay(), 3) / iters


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    assert torch.cuda.is_available(), "needs a GPU"
    print(card())
    print("SMs: %d" % torch.cuda.get_device_properties(0).multi_processor_count)
    for name, t_count, m in WORKLOADS:
        base = make(t_count, m, seed=t_count + m)
        per_copy = sum(v.numel() * v.element_size() for v in base.values())
        copies = max(1, math.ceil(3 * L2 / per_copy))
        xs = [base] + [make(t_count, m, seed=t_count + m + k) for k in range(1, copies)]
        for mode in ("gae", "returns", "vtrace"):
            err = check(mode, base, call(mode, base))
            ws = postprocess._lib.lib.ssd_advantages_workspace_bytes(t_count, m)
            times, ttimes = [], []
            iters = max(3, int(2e9 / algorithmic_bytes(mode, t_count, m)))
            titers = 1 if t_count * m > 5e7 else 3
            for _ in range(rounds):
                call(mode, xs[0])
                torch.cuda.synchronize()
                times.append(events(lambda i: call(mode, xs[i % copies]), iters))
                torch_loop(mode, xs[0])
                torch.cuda.synchronize()
                ttimes.append(events(lambda i: torch_loop(mode, xs[i % copies]), titers))
            med, tmed = float(np.median(times)), float(np.median(ttimes))
            if t_count * m <= 2e7:   # small calls: also without the per-call host work (inputs stay in L2 here)
                print("(%s) T=%d M=%d %-7s in one CUDA graph of 50 calls on one input set: %.4f ms per call"
                      % (name, t_count, m, mode, graphed(mode, xs[0], 50)), flush=True)
            nbytes = algorithmic_bytes(mode, t_count, m)
            print("(%s) T=%d M=%d %-7s kernel %.4f ms [%.4f, %.4f]  %.2f TB/s = %.0f %% of 7.7 TB/s  torch loop %.2f ms [%.2f, %.2f]"
                  "  speedup %.0fx  max err vs oracle %.2e  workspace %d B  copies %d"
                  % (name, t_count, m, mode, med, min(times), max(times), nbytes / med / 1e9, 100 * nbytes / med / 1e3 / PEAK * 1e6,
                     tmed, min(ttimes), max(ttimes), tmed / med, err, ws, copies), flush=True)
        del xs, base
        torch.cuda.empty_cache()
    if "--profile" in sys.argv:
        from torch.profiler import ProfilerActivity, profile
        x = make(1000, 327680, seed=1)
        for mode in ("gae", "returns", "vtrace"):
            call(mode, x)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for mode in ("gae", "returns", "vtrace"):
                for _ in range(3):
                    call(mode, x)
            torch.cuda.synchronize()
        print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=12))


if __name__ == "__main__":
    main()
