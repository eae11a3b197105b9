"""Times MOANet.step (ssd_moa_step: the model of other agents, its A counterfactuals and the social-influence reward in one
kernel) against the torch route it replaces, on the trunk features of 65 536 envs x 5 agents = 327 680 agents per call:
  harvest  A = 8, cleanup  A = 9, each with one shared MOA and with one MOA per agent id (P = N = 5).
  kernel   MOANet.step without and with the [M, A, N-1, A] counterfactual logits written;
  torch    A + 1 MOA steps in torch: bf16 gate GEMMs ([x | one-hot] W + h U), ssd_policy_lstm_cell, the bf16 head GEMM, then
           softmax, marginal and KL over [M, A, N-1, A] in fp32 (per-agent weights as batched GEMMs over the N agent ids).
The torch route is first checked against the kernel at this size (max abs difference of pred, h' and the influence; bf16
operands).  Then alternating rounds, median [min, max] ms per call (CUDA events around `iters` back-to-back calls); the card's
name, power limit and max SM clock are read in the same run.  The recurrent state (2 x 168 MB in, 2 x 168 MB out) does not fit
the 126 MB L2.  Run on a GPU: python profiles/moa_bench.py [num_envs] [rounds]"""
import ctypes as C
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from sequential_social_dilemma_games_b200 import _lib, policy  # noqa: E402
from sequential_social_dilemma_games_b200.batched import BatchedSSDEnv, make_config  # noqa: E402


def timed(fn, iters, warm=2):
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
        q = "not readable (%s)" % e
    return "%s, power limit, max SM clock: %s" % (name, q)


class TorchMOA(object):
    """The torch route: weights [P, K, 512] etc. in bf16, agents grouped by weight set as [P, M / P, ...]."""

    def __init__(self, sets, n, a):
        dev = lambda k, dt: torch.stack([torch.from_numpy(ws[k]) for ws in sets]).to("cuda", dtype=dt)
        self.w, self.u, self.wl = dev("moa_lstm_w", torch.bfloat16), dev("moa_lstm_u", torch.bfloat16), dev("moa_logits_w", torch.bfloat16)
        self.b, self.bl = dev("moa_lstm_b", torch.float32), dev("moa_logits_b", torch.float32)
        self.n, self.a, self.p = n, a, len(sets)
        self.others = [[j for j in range(n) if j != i] for i in range(n)]

    def _group(self, t):   # agent-major [M, ...] -> [P, M / P, ...]
        return t.reshape(-1, self.p, *t.shape[1:]).transpose(0, 1) if self.p > 1 else t[None]

    def step(self, x, joint, pl, h, c):
        n, a, m = self.n, self.a, x.shape[0]
        joint = joint.long().reshape(-1, n)
        oh = torch.nn.functional.one_hot(joint.clamp(0, a - 1), a).to(torch.bfloat16) * ((joint >= 0) & (joint < a))[..., None]   # [B, N, A]
        idx = torch.arange(m, device="cuda")
        i = idx % n
        oth = torch.stack([torch.tensor(self.others[k], device="cuda") for k in range(n)])[i]   # [M, N-1]
        others = oh[idx[:, None] // n, oth].reshape(m, (n - 1) * a)
        own_actual = oh.reshape(m, a)
        h16 = self._group(h.to(torch.bfloat16))
        hu = torch.bmm(h16, self.u)   # [P, M/P, 512]
        outs = []
        for ap in range(a + 1):   # ap = a: the actual joint action
            own = own_actual if ap == a else torch.nn.functional.one_hot(torch.full((m,), ap, device="cuda"), a).to(torch.bfloat16)
            inp = self._group(torch.cat([x.to(torch.bfloat16), own, others], dim=1))
            gates = torch.baddbmm(hu, inp, self.w)   # bf16 [P, M/P, 512], bias added in the cell kernel
            hn, cn = torch.empty_like(h), torch.empty_like(c)
            h16n = torch.empty((self.p, m // self.p, 128), dtype=torch.bfloat16, device="cuda")
            gp = gates.contiguous()
            cg = self._group(c).contiguous()
            cn_g, hn_g = torch.empty_like(cg), torch.empty_like(cg)
            st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            for q in range(self.p):
                _lib.check(_lib.lib.ssd_policy_lstm_cell(C.c_void_p(gp[q].data_ptr()), C.c_void_p(self.b[q].data_ptr()),
                                                         C.c_void_p(cg[q].data_ptr()), C.c_void_p(cn_g[q].data_ptr()),
                                                         C.c_void_p(hn_g[q].data_ptr()), C.c_void_p(h16n[q].data_ptr()), m // self.p, 128, st))
            y = (torch.bmm(h16n, self.wl).float() + self.bl[:, None]).transpose(0, 1).reshape(m, n - 1, a) if self.p > 1 \
                else (torch.bmm(h16n, self.wl).float() + self.bl[:, None])[0].reshape(m, n - 1, a)
            outs.append(y)
            if ap == a:
                hn = hn_g.transpose(0, 1).reshape(m, 128) if self.p > 1 else hn_g[0]
                cn = cn_g.transpose(0, 1).reshape(m, 128) if self.p > 1 else cn_g[0]
        pred, cf = outs[a], torch.stack(outs[:a], dim=1)   # [M, A, N-1, A]
        pi = torch.softmax(pl, dim=1)
        q = torch.einsum("ma,makx->mkx", pi, torch.softmax(cf, dim=-1))
        q = q / q.sum(dim=-1, keepdim=True)
        logp = torch.log_softmax(pred, dim=-1)
        ipa = torch.where(logp.exp() > 0, logp.exp() * (logp - q.log()), torch.zeros_like(logp)).sum(dim=-1)
        return pred, ipa.sum(dim=1), ipa, hn, cn


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    N, M = 5, B * 5
    print(card())
    print("%d envs x %d agents = %d agents per call, %d alternating rounds" % (B, N, M, rounds))
    for game, A in (("harvest", 8), ("cleanup", 9)):
        env = BatchedSSDEnv(make_config(game, num_agents=N), B, seed=1)
        obs = env.reset()
        pnet = policy.ConvToFCNet(policy.random_weights(num_outputs=A, seed=0))
        x = pnet.features(obs)
        h0, c0 = pnet.initial_state(M)
        st = pnet.policy_step(obs, h0, c0)
        joint, pl = st.actions.view(B, N), st.logits
        g = torch.Generator(device="cuda").manual_seed(2)
        h_rows = 0.5 * torch.randn((M, 128), device="cuda", generator=g)
        c_rows = 0.5 * torch.randn((M, 128), device="cuda", generator=g)
        env.close()
        pnet.close()
        for kind in ("shared", "per_agent"):
            sets = [policy.random_moa_weights(N, A, seed=10 + k) for k in range(N if kind == "per_agent" else 1)]
            net = policy.MOANet(sets if kind == "per_agent" else sets[0], N)
            ref = TorchMOA(sets, N, A)
            h, c = net.state_from_rows(h_rows), net.state_from_rows(c_rows)
            s = net.step(x, joint, pl, h, c)
            pr, infl, _, hr, _ = ref.step(x, joint, pl, h_rows, c_rows)
            torch.cuda.synchronize()
            d_pred = (s.pred - pr).abs().max().item()
            d_h = (net.state_rows(s.h, M) - hr).abs().max().item()
            d_inf = (s.influence - infl).abs().max().item()
            print("%s %s: torch route vs kernel, max abs diff pred %.3g, h' %.3g, influence %.3g (mean influence %.4g)"
                  % (game, kind, d_pred, d_h, d_inf, s.influence.mean().item()))
            assert d_pred < 5e-2 and d_h < 5e-2 and d_inf < 5e-2, "the torch route disagrees with the kernel"
            variants = {"kernel": lambda: net.step(x, joint, pl, h, c),
                        "kernel+cf": lambda: net.step(x, joint, pl, h, c, counterfactuals=True),
                        "torch": lambda: ref.step(x, joint, pl, h_rows, c_rows)}
            iters = {"kernel": 20, "kernel+cf": 20, "torch": 3}
            times = {k: [] for k in variants}
            for _ in range(rounds):
                for k, fn in variants.items():
                    times[k].append(timed(fn, iters[k]))
            for k, ts in times.items():
                ts = sorted(ts)
                print("  %-10s median %.3f ms [%.3f, %.3f]" % (k, ts[len(ts) // 2], ts[0], ts[-1]))
            med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
            print("  torch / kernel: %.2fx" % (med["torch"] / med["kernel"]))
            net.close()
            del ref
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
