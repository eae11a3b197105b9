#!/usr/bin/env python
"""Benchmark of the SSD gridworld step path (BASELINE.json: Harvest agent-steps/sec incl. obs).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one MapEnv.step over the whole batch of synthetic-action environments resident on a
GPU (one fused kernel launch).  Workload at N=1: BASELINE.json configs[2] -- HarvestEnv, 5 agents,
default HARVEST_MAP, 65 536 batched envs, 15x15x3 egocentric uint8 observations; with N>1 every GPU
owns 65 536 envs of its own (weak scaling, no collective on the step path, Philox streams keyed by
global env id).  Prints ONE JSON line (rank 0).

`value` times K steps of BatchedSSDEnv.step with consecutive steps chained (SSD_OPT_CHAIN_STEPS: programmatic dependent
launch; the actions are pre-generated, which is the option's precondition); `stream_ordered` is the same K steps
without chaining (what a policy in the loop gets); `rollout` (configs only) is ssd_rollout, one C call for T scripted steps; `e2e` goes through ssd_step_host with pinned host buffers (H2D actions,
D2H observations + rewards inside the timed region) next to a measured host-copy roof; `configs` carries the other
BASELINE.json configurations (Cleanup, the tiled 10-agent stress map, the strong split of 65 536 envs over the GPUs);
`cpu_baseline` / `--impl reference` time the C port of the reference's step on the host cores, and
`cpu_baseline.python_reference` the reference's own unmodified Python step, one process per core.

`--dump-outputs DIR` writes what the last timed step returned (rank 0): DIR/obs.npy and DIR/reward.npy, float32, for a
fixed seeded sample of the envs.  The inputs depend on the arguments only, so two builds run with the same arguments can be
compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "harvest_agent_steps_per_sec_obs_incl"
UNIT = "agent-steps/s"
HORIZON = 1000  # RLlib "horizon" of the reference's training configs (train_baseline.py:131)
BURN_IN = 100   # untimed steps between a reset and the first timed step: right after reset() the agents still stand crowded
                # around the spawn points (move conflicts in most envs) and the orchard is full, which is not what the other
                # 900 steps of an episode look like; a short timed region would otherwise sample only that stretch


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=65536)
    ap.add_argument("--game", default="harvest", choices=["harvest", "cleanup"])
    ap.add_argument("--agents", type=int, default=5)
    ap.add_argument("--view", type=int, default=7)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--cpu-sample-envs", type=int, default=8192)
    ap.add_argument("--config-steps", type=int, default=1000, help="timed steps of every entry of the `configs` array")
    ap.add_argument("--pyref-steps", type=int, default=1000, help="steps of the Python reference per process (BASELINE.md section 4)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the batch-size x view-radius sweep (BASELINE.json configs[4])")
    ap.add_argument("--sweep-steps", type=int, default=60)
    ap.add_argument("--no-chain", action="store_true", help="stream-ordered steps only (no programmatic dependent launch)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the observations and rewards of the last timed step to DIR as "
                                                          "float32 .npy files (a fixed seeded sample of the envs, at most 64 MB)")
    return ap.parse_args()


DUMP_ENVS = 1024        # envs in a --dump-outputs sample: 1024 x 5 agents x 15x15x3 observations are 14 MB as float32
DUMP_BYTES = 60 << 20   # cap for larger agent counts and views


def dump_index(num_envs, values_per_env):
    """Sorted env rows of the --dump-outputs sample; depends on the batch shape only."""
    import numpy as np
    k = max(1, min(num_envs, DUMP_ENVS, DUMP_BYTES // (4 * values_per_env)))
    return np.sort(np.random.RandomState(0).choice(num_envs, k, replace=False))


def dump_outputs(out_dir, **arrays):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float32))


def workload(args):
    """config of the JSON line; both arms print the same keys (the reference arm runs a bounded sample of it on the CPU)."""
    return {"workload": "%sEnv %d agents, default map, %d batched envs per GPU, %dx%dx3 uint8 egocentric obs, "
                        "uniform random actions, horizon %d" % (args.game.capitalize(), args.agents, args.envs_per_gpu,
                                                                2 * args.view + 1, 2 * args.view + 1, HORIZON),
            "game": args.game, "num_agents": args.agents, "envs_per_gpu": args.envs_per_gpu,
            "view_radius": args.view, "rng": "philox4x32-10 (production mode)",
            "actions": "pre-generated on device, ring of 16 x [B,N] int8",
            "episode": "reset every %d steps; timed regions start at least %d untimed steps after a reset (W warm-up steps included)" % (HORIZON, BURN_IN),
            "l2": "per-step working set (state r/w + obs write) is %.0f MB > 126 MB L2; no explicit flush"
                  % ((2 * 608 + 3 * args.agents * (2 * args.view + 1) ** 2) * args.envs_per_gpu / 1e6),
            "parallelism": "env-sharded x%d" % args.gpus}


# ---------------------------------------------------------------------------------- clocks
class ClockSampler(object):
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self._stop, self._th = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        self._th = threading.Thread(target=self._run, daemon=True)
        self._th.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._th.join(timeout=10)
        return False

    def mark(self):
        return len(self.rows)

    def summary(self, n_timed=None):
        sm, reasons, mx = [], set(), None
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "samples_in_timed_regions": n_timed,
                "how": "nvidia-smi polled every 50 ms over the two timed regions and, because K steps can be shorter than one poll, "
                       "over a further >= 1.5 s loop of the same step kernel right after them"}


# ---------------------------------------------------------------------------------- CPU baselines
def cpu_port_rate(args, seconds_target, steps=None, warmup=2, dump_dir=None):
    """Times oracle/ssd_oracle.c (the CPU port of the reference's step path) on the host cores on a
    bounded sample of the same workload.  Returns (agent-steps/s, cores, sample description, ms/step)."""
    import numpy as np
    from oracle.oracle import OracleEnv
    from sequential_social_dilemma_games_b200.config import make_config  # config only: never loads libssd_b200.so
    cores = min(os.cpu_count() or 1, 256)
    cfg = make_config(args.game, num_agents=args.agents, view_size=args.view)
    B = args.cpu_sample_envs
    env = OracleEnv(cfg, B, seed=0, n_threads=cores)
    env.reset(render=False)
    rng = np.random.RandomState(0)
    ring = rng.randint(cfg.num_actions, size=(16, B, cfg.num_agents)).astype(np.int8)
    buf = env._new_obs()
    for i in range(warmup):
        env.step(ring[i % 16], obs_out=buf)
    n, t0 = 0, time.perf_counter()
    while True:
        _, rew = env.step(ring[n % 16], obs_out=buf)
        n += 1
        dt = time.perf_counter() - t0
        if (steps is not None and n >= steps) or (steps is None and dt >= seconds_target):
            break
    if dump_dir:
        idx = dump_index(B, buf[0].size + cfg.num_agents)
        dump_outputs(dump_dir, obs=buf[idx], reward=rew[idx])
    rate = n * B * cfg.num_agents / dt
    sample = ("%d envs x %d steps of the same workload (%sEnv, %d agents, %dx%dx3 obs, uniform random actions), "
              "oracle/ssd_oracle.c, %d pthreads" % (B, n, args.game.capitalize(), cfg.num_agents, cfg.view_width, cfg.view_width, cores))
    return rate, cores, sample, dt / n * 1e3


SURVEY_PYTHON_FIGURE = {"per_process_agent_steps_per_s": 1342.0, "aggregate_agent_steps_per_s": 10565.0, "cores": 8,
                        "note": "NOT measured in this run: SURVEY.md section 6 / BASELINE.md section 2, unmodified reference on the 8-vCPU "
                                "build container"}


def python_reference_rate(args):
    """The reference's OWN Python MapEnv.step (map_env.py:152), unmodified, one process per host core (BASELINE.md section 4,
    SURVEY.md 8d config 1).  The tree comes from $SSD_REFERENCE_ROOT, /root/reference or baseline/_ref (first that exists;
    baseline/_ref is what __graft_entry__.build() copies verbatim in the build container and what travels to the GPU box)."""
    roots = [os.environ.get("SSD_REFERENCE_ROOT"), "/root/reference", os.path.join(ROOT, "baseline", "_ref")]
    root = next((r for r in roots if r and os.path.isdir(os.path.join(r, "social_dilemmas", "envs"))), None)
    if root is None:
        return {"unavailable": "no reference tree at $SSD_REFERENCE_ROOT, /root/reference or baseline/_ref", "survey_figure": SURVEY_PYTHON_FIGURE}
    cores = os.cpu_count() or 1
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "pyref_worker.py"), "--root", root, "--game", args.game,
           "--agents", str(args.agents), "--view", str(args.view), "--steps", str(args.pyref_steps)]
    env = dict(os.environ, OMP_NUM_THREADS="1", OPENBLAS_NUM_THREADS="1", MKL_NUM_THREADS="1")
    t0 = time.perf_counter()
    procs = [subprocess.Popen(cmd + ["--seed", str(s)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env)
             for s in range(cores)]
    rates, errs = [], []
    for p in procs:
        try:
            out, err = p.communicate(timeout=600)
            rates.append(json.loads(out.strip().splitlines()[-1])["agent_steps_per_s"])
        except Exception as exc:  # noqa: BLE001
            p.kill()
            errs.append(repr(exc)[:120])
    if not rates:
        return {"unavailable": "every worker failed: %s" % "; ".join(errs[:2]), "survey_figure": SURVEY_PYTHON_FIGURE}
    return {"per_process_agent_steps_per_s": sum(rates) / len(rates), "aggregate_agent_steps_per_s": sum(rates),
            "unit": UNIT, "cores": cores, "processes": len(rates), "failed": len(errs), "wall_s": time.perf_counter() - t0,
            "kind": "reference", "root": os.path.relpath(root, ROOT) if root.startswith(ROOT) else root,
            "sample": "unmodified %sEnv(num_agents=%d), default map, view radius %d: reset() + %d steps of MapEnv.step with uniform "
                      "random actions per process, seeds 0..%d, only env.step timed (BASELINE.md section 4)"
                      % (args.game.capitalize(), args.agents, args.view, args.pyref_steps, cores - 1)}


def cpu_baseline(args, seconds_target=12.0, steps=None, warmup=2, dump_dir=None):
    rate, cores, sample, ms = cpu_port_rate(args, seconds_target, steps=steps, warmup=warmup, dump_dir=dump_dir)
    base = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
    try:
        base["python_reference"] = python_reference_rate(args)
    except Exception as exc:  # noqa: BLE001
        base["python_reference"] = {"unavailable": repr(exc)[:200], "survey_figure": SURVEY_PYTHON_FIGURE}
    return base, ms


def run_reference(args, rank):
    """--impl reference: the reference's step path on the host cores: its C port (oracle/ssd_oracle.c, pinned to the
    reference's golden outputs) with all host threads is the line's value -- the stronger CPU baseline -- and the reference's
    own Python step, one process per core, is reported inside cpu_baseline.python_reference.  Never touches libssd_b200.so."""
    if rank != 0:
        return
    base, ms = cpu_baseline(args, steps=args.steps, warmup=max(args.warmup, 1), dump_dir=args.dump_outputs)
    rate = base["value"]
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic", "config": workload(args),
            "cpu_baseline": base,
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------- our arm
def run_ours(args, rank, world, local_rank):
    import numpy as np  # noqa: F401
    import torch
    import torch.distributed as dist
    from sequential_social_dilemma_games_b200.batched import BatchedSSDEnv
    from sequential_social_dilemma_games_b200.config import make_config
    from sequential_social_dilemma_games_b200.maps import CLEANUP_MAP, tile_map

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks, peak_src = {}, "fallback 6650 GB/s (B200_PROFILING.md)"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
        peak_src = "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    class Run(object):
        """One workload on this rank: env, action ring, output buffers, the step loop with RLlib's horizon."""

        def __init__(self, cfg, B, env_id_offset):
            self.cfg, self.B, self.N = cfg, B, cfg.num_agents
            self.env = BatchedSSDEnv(cfg, B, device=dev, seed=0, env_id_offset=env_id_offset)
            g = torch.Generator(device=dev).manual_seed(1234 + rank)
            self.ring = torch.randint(0, cfg.num_actions, (16, B, self.N), generator=g, device=dev, dtype=torch.int8)
            self.obs = torch.empty(self.env.obs_shape, dtype=torch.uint8, device=dev)
            self.rew = torch.empty((B, self.N), dtype=torch.int32, device=dev)
            self.n = 0

        def one_step(self):
            if self.n % HORIZON == 0:
                self.env.reset(out=self.obs)  # episode boundary, as RLlib's horizon does
            self.env.step(self.ring[self.n % 16], out=self.obs, reward_out=self.rew)
            self.n += 1

        def timed(self, n):
            """(this rank's ms, max over ranks ms) of n steps; device-timed, barrier + synchronize on both sides."""
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            e0.record()
            for _ in range(n):
                self.one_step()
            e1.record()
            barrier()
            ms = e0.elapsed_time(e1)
            return ms, max_ranks(ms)

        def measure(self, steps, warmup, chain=True):
            """stream-ordered, chained and ssd_rollout timings -> dict for the JSON line.  Every mode starts from a fresh episode
            (reset + `warmup` steps), so that all of them see the same stretch of it: Cleanup gets slower as waste is cleaned."""
            def fresh():
                self.n = 0
                for _ in range(warmup):
                    self.one_step()
            fresh()
            _, ms_plain = self.timed(steps)
            out = {"stream_ordered": {"ms_per_step": ms_plain / steps}}
            if chain:
                self.env.chain_steps(True)
                fresh()
                _, ms_max = self.timed(steps)
                self.env.chain_steps(False)
                out["chained"] = {"ms_per_step": ms_max / steps}
                fresh()
                out["rollout"] = self.rollout_ms(min(steps, 400))
            return out

        def rollout_ms(self, T):
            """ssd_rollout: T steps whose actions all exist up front, one C call (one launch of the wide kernel for batches below
            half a wave of CTAs, chained launches otherwise).  No episode reset inside (T <= 400)."""
            acts = self.ring.repeat((T + 15) // 16, 1, 1)[:T].contiguous()
            ring = self.obs.unsqueeze(0)
            rews = torch.empty((T, self.B, self.N), dtype=torch.int32, device=dev)
            self.env.rollout(acts[:8], ring, rews[:8])
            l0 = self.env.launch_count
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            e0.record()
            self.env.rollout(acts, ring, rews)
            e1.record()
            barrier()
            ms = max_ranks(e0.elapsed_time(e1))
            self.n += T + 8
            return {"ms_per_step": ms / T, "steps": T,
                    "launches": "one launch for all steps (wide kernel)" if self.env.launch_count - l0 == 1 else "one chained launch per step"}

        def close(self):
            self.env.close()

    # ------------------------------------------------------------------ headline: BASELINE.json configs[2], weak scaling
    cfg = make_config(args.game, num_agents=args.agents, view_size=args.view)
    B, N = args.envs_per_gpu, cfg.num_agents
    run = Run(cfg, B, rank * B)
    env = run.env
    for _ in range(max(args.warmup, BURN_IN)):
        run.one_step()
    with ClockSampler(local_rank) as clk:  # clocks and throttle reasons over both timed regions
        # stream-ordered steps first (every kernel waits for the previous one to drain) ...
        _, ms_plain = run.timed(args.steps)
        # ... then the headline: consecutive steps chained with programmatic dependent launch (SSD_OPT_CHAIN_STEPS).
        # The actions are pre-generated, which is the option's precondition; results are identical (tests/test_gpu_parity.py).
        chained = not args.no_chain
        if chained:
            env.chain_steps(True)
            for _ in range(args.warmup):
                run.one_step()
        launches0 = env.launch_count
        ms, ms_max = run.timed(args.steps)
        launches = env.launch_count - launches0  # kernels of the timed region: one fused step kernel per step (+ 2 per episode reset)
        n_timed = clk.mark()
        if args.dump_outputs and rank == 0:  # now: the clocks loop below steps on in the same buffers
            sel = torch.from_numpy(dump_index(B, run.obs[0].numel() + N)).to(dev)
            dump_outputs(args.dump_outputs, obs=run.obs[sel].cpu().numpy(), reward=run.rew[sel].cpu().numpy())
        # K steps can be shorter than one nvidia-smi poll: keep the same kernel running for >= 1.5 s so that the clocks line
        # describes the GPU under this load (not part of any reported time)
        t_end = time.perf_counter() + 1.5
        while time.perf_counter() < t_end:
            for _ in range(200):
                run.one_step()
            torch.cuda.synchronize(dev)
    value = world * B * N * args.steps / (ms_max * 1e-3)
    env.chain_steps(False)
    clocks = clk.summary(n_timed)

    # ------------------------------------------------------------------ end to end through the C-ABI with HOST buffers
    e2e = None
    if not args.no_e2e:
        ring_host = torch.empty((16, B, N), dtype=torch.int8, pin_memory=True)
        ring_host.copy_(run.ring.cpu())
        o_host = torch.empty(env.obs_shape, dtype=torch.uint8, pin_memory=True)
        r_host = torch.empty((B, N), dtype=torch.int32, pin_memory=True)
        a_np, o_np, r_np = ring_host.numpy(), o_host.numpy(), r_host.numpy()
        for i in range(3):
            env.step_host(a_np[i % 16], obs_host=o_np, reward_host=r_np)
        barrier()
        t0 = time.perf_counter()
        for i in range(args.e2e_steps):
            env.step_host(a_np[i % 16], obs_host=o_np, reward_host=r_np)
        torch.cuda.synchronize(dev)
        dt = max_ranks(time.perf_counter() - t0)
        d2h = B * (cfg.num_agents * cfg.view_width ** 2 * 3 + 4 * N)
        # the roof of that path: what the host side of this box takes when every rank copies the same bytes device -> pinned host
        # at the same time, nothing else running (eight chunks per step on two streams, as ssd_step_host issues them)
        dsrc = torch.empty(d2h, dtype=torch.uint8, device=dev)
        hdst = torch.empty(d2h, dtype=torch.uint8, pin_memory=True)
        chunks = [(i * d2h // 8, (i + 1) * d2h // 8) for i in range(8)]
        streams = [torch.cuda.Stream(dev), torch.cuda.Stream(dev)]

        def copy_once():
            for k, (lo, hi) in enumerate(chunks):
                with torch.cuda.stream(streams[k & 1]):
                    hdst[lo:hi].copy_(dsrc[lo:hi], non_blocking=True)
            for s in streams:
                s.synchronize()
        for _ in range(3):
            copy_once()
        barrier()
        t0 = time.perf_counter()
        for _ in range(10):
            copy_once()
        roof_dt = max_ranks(time.perf_counter() - t0) / 10
        roof_gbs = world * d2h / roof_dt / 1e9
        achieved_gbs = world * d2h * args.e2e_steps / dt / 1e9
        e2e = {"value": world * B * N * args.e2e_steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": B * N, "d2h_bytes_per_step": d2h,
               "api": "ssd_step_host (pinned host buffers: int8 actions in, uint8 obs + int32 rewards out)",
               "steps": args.e2e_steps, "achieved_gbs": achieved_gbs, "roof_gbs": roof_gbs, "frac_of_roof": achieved_gbs / roof_gbs,
               "roof": "device -> pinned host copy of the same bytes per step, all %d ranks at once, nothing else running "
                       "(cudaMemcpyAsync, 8 chunks on 2 streams), measured in this run" % world}
        del dsrc, hdst

    stats = env.stats()
    tot = torch.tensor([stats["env_steps"], stats["reward_sum"], stats["apples_eaten"], stats["hits"]],
                       dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(tot)  # the only collective: end-of-run stats

    # informational: the same step with its consumer on the device (policy forward pass + sampled actions, no PCIe).  Not
    # the contract's e2e; harvest r = 7 only (the trunk kernel is built for 15x15 observations); never fatal.
    on_device = None
    if rank == 0 and args.view == 7 and not args.no_e2e:
        try:
            from sequential_social_dilemma_games_b200 import policy
            net = policy.ConvToFCNet(policy.random_weights(num_outputs=cfg.num_actions, seed=0), device=dev)
            st = {"obs": env.reset(), "hc": net.initial_state(B * N)}

            def loop_step():
                a, _, h, c = net.act(st["obs"].reshape(-1, 15, 15, 3), *st["hc"])
                st["hc"] = (h, c)
                st["obs"], _ = env.step(a.reshape(B, N))
            for _ in range(5):
                loop_step()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(20):
                loop_step()
            e1.record()
            torch.cuda.synchronize(dev)
            ms_loop = e0.elapsed_time(e1) / 20
            on_device = {"value": B * N / (ms_loop * 1e-3), "unit": UNIT, "ms_per_step": ms_loop, "n_gpus": 1,
                         "what": "env.step + ConvToFCNet.act (tcgen05 trunk kernel, tcgen05 LSTM + heads + Gumbel-max sampling kernel); "
                                 "observations and actions never leave the device; random-init weights"}
            net.close()
        except Exception as exc:  # noqa: BLE001
            on_device = {"unavailable": repr(exc)[:200]}
    alg = env.algorithmic_bytes_per_env_step
    envs_per_cta = env.envs_per_cta
    run.close()
    del run, env

    # ------------------------------------------------------------------ the other BASELINE.json configurations (informational)
    configs = []
    if not args.no_configs:
        tiled = tile_map(CLEANUP_MAP)
        plan = [
            ("BASELINE.json configs[2] as written: HarvestEnv 5 agents, 65 536 envs TOTAL split over the GPUs (strong scaling)",
             "harvest", 5, None, max(65536 // world, 1), "strong", 65536 // world * world),
            ("CleanupEnv 5 agents, default map, 65 536 envs per GPU", "cleanup", 5, None, 65536, "weak", 65536 * world),
            ("BASELINE.json configs[3]: CleanupEnv 10 agents on the 2x2-tiled map (50x36), 16 384 envs per GPU, P(FIRE) = P(CLEAN) = 0.25",
             "cleanup", 10, tiled, 16384, "weak", 16384 * world),
        ]
        for name, game, n_ag, amap, b_rank, scaling, b_total in plan:
            try:
                c = make_config(game, num_agents=n_ag, view_size=7, ascii_map=amap)
                r = Run(c, b_rank, rank * b_rank)
                if amap is not None:  # the stress mix of SURVEY 8d config 4: a quarter FIRE, a quarter CLEAN, the rest uniform over 0..6
                    g = torch.Generator(device=dev).manual_seed(99 + rank)
                    u = torch.rand((16, b_rank, n_ag), generator=g, device=dev)
                    base = torch.randint(0, 7, (16, b_rank, n_ag), generator=g, device=dev, dtype=torch.int8)
                    r.ring = torch.where(u < 0.25, torch.full_like(base, 7), torch.where(u < 0.5, torch.full_like(base, 8), base))
                m = r.measure(args.config_steps, min(args.warmup, 30), chain=not args.no_chain)
                a_bytes = r.env.algorithmic_bytes_per_env_step
                entry = {"name": name, "game": game, "num_agents": n_ag, "envs_per_gpu": b_rank, "envs_total": b_total, "scaling": scaling,
                         "steps": args.config_steps, "algorithmic_bytes_per_env_step": a_bytes}
                for k in ("stream_ordered", "chained", "rollout"):
                    if k in m:
                        ms_k = m[k]["ms_per_step"]
                        gbs = a_bytes * b_rank / (ms_k * 1e-3) / 1e9
                        entry[k] = {"ms_per_step": ms_k, "value": b_total * n_ag / (ms_k * 1e-3), "unit": UNIT,
                                    "roofline_frac_per_gpu": gbs / peak, "achieved_gbs_per_gpu": gbs}
                        if k == "rollout":
                            entry[k]["launches"] = m[k]["launches"]
                configs.append(entry)
                r.close()
                del r
            except Exception as exc:  # noqa: BLE001
                configs.append({"name": name, "unavailable": repr(exc)[:200]})

    # ------------------------------------------------------------------ BASELINE.json configs[4]: batch size x view radius (informational)
    sweep = []
    if not args.no_sweep:
        for r_view in (5, 7, 10):
            for b_rank in (1024, 16384, 262144, 1048576):
                try:
                    c = make_config("harvest", num_agents=5, view_size=r_view)
                    r = Run(c, b_rank, rank * b_rank)
                    for _ in range(20):
                        r.one_step()
                    _, ms_sw = r.timed(args.sweep_steps)
                    ms_sw /= args.sweep_steps
                    a_bytes = r.env.algorithmic_bytes_per_env_step
                    sweep.append({"envs_per_gpu": b_rank, "view_radius": r_view, "ms_per_step": ms_sw,
                                  "value": world * b_rank * 5 / (ms_sw * 1e-3),
                                  "roofline_frac_per_gpu": a_bytes * b_rank / (ms_sw * 1e-3) / 1e9 / peak})
                    r.close()
                    del r
                    torch.cuda.empty_cache()
                except Exception as exc:  # noqa: BLE001
                    sweep.append({"envs_per_gpu": b_rank, "view_radius": r_view, "unavailable": repr(exc)[:160]})

    if rank == 0:
        kernel_ms = ms / args.steps  # this rank's average step-kernel launch (one launch per step)
        achieved = alg * B / (kernel_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                tj = json.load(f)
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source", "profiles/traffic.json")
        except Exception:
            pass
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic", "config": workload(args),
                "launch": {"envs_per_cta": envs_per_cta,
                           "step_launch": "chained: programmatic dependent launch, per-warp completion words (SSD_OPT_CHAIN_STEPS)"
                           if chained else "stream-ordered"},
                "stream_ordered": {"value": world * B * N * args.steps / (ms_plain * 1e-3), "ms_per_step": ms_plain / args.steps,
                                   "roofline_frac": alg * B / (ms_plain / args.steps * 1e-3) / 1e9 / peak,
                                   "note": "same K steps without chaining: every step kernel drains before the next starts (what a policy in the loop gets)"},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic,
                             "traffic_source": "NOT measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of one launch from the committed "
                                               "`ncu --set full` capture (%s)" % traffic_src,
                             "kernel": "ssd_step_fast_kernel<%s,philox,V=%d>" % (args.game.upper(), 2 * args.view + 1), "peak_source": peak_src,
                             "algorithmic_bytes_per_env_step": alg, "units_per_launch": B},
                "clocks": clocks, "gpu_launches": launches, "e2e": e2e,
                "totals": {"env_steps": int(tot[0]), "reward_sum": int(tot[1]), "apples_eaten": int(tot[2]), "hits": int(tot[3])}}
        if configs:
            line["configs"] = configs
        if sweep:
            line["sweep"] = {"what": "BASELINE.json configs[4]: HarvestEnv 5 agents, stream-ordered steps, envs per GPU x view radius, "
                                     "%d timed steps each; value = all GPUs together (weak scaling)" % args.sweep_steps,
                             "unit": UNIT, "rows": sweep}
        if on_device is not None:
            line["on_device_loop"] = on_device
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"], _ = cpu_baseline(args, 12.0)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
