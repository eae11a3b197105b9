"""Generates tests/golden/*.npz by running the UNMODIFIED Python reference at /root/reference.

Run in the build container only (the reference tree does not exist on the GPU box):

    python tests/golden/make_golden.py

Two kinds of fixtures (SURVEY.md section 8c):
  *_tape.npz    "tape-out": the reference runs on its own MT19937 streams
                (np.random.seed(s); random.seed(s)); the move order, every np.random.rand value
                and the shuffled waste order are recorded per step and replayed into the
                implementation under test.
  *_philox.npz  "Philox-in": np.random.shuffle / rand / randint and random.shuffle are
                replaced by the production Philox streams (oracle/ref_harness.PhiloxIn), so the
                implementation under test generates its own draws, reset() included.

Every fixture stores the initial state, the actions, and after EVERY step the reference's
grid, positions, orientations, rewards and uint8 observations (the float64 observation is
(u8 - 128.0) / 255.0 exactly; ref_harness.obs_u8 asserts that).

The Cleanup tapes (seeded=True) are "seeded tapes": instead of megabytes of incompressible uniform doubles and
shuffled waste orders they store the MT19937 states of np.random / random right after reset();
tests/golden_util.py regenerates the tape from them (the draw counts per step are stored, and this script
asserts that the regenerated tape equals the recorded one).  Where an env never shuffles its waste list within
the recorded steps, the recording does not determine the state of `random`; any state replays the same tape.
Observations are kept every `obs_every`-th step, everything else every step.  Fixtures are LZMA-compressed
.npz files (np.load reads them), so that each stays below 1 MB.
"""
import io
import os
import random
import sys
import zipfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import ref_harness as rh  # noqa: E402
from sequential_social_dilemma_games_b200.config import (  # noqa: E402
    EnvConfig, KIND_CLEANUP, KIND_HARVEST)
from sequential_social_dilemma_games_b200.maps import CLEANUP_MAP, HARVEST_MAP, tile_map  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
DENSE_MAP = ['@@@@@@@', '@PPPPA@', '@PPAAA@', '@AAPPP@', '@PPPPP@', '@@@@@@@']


def make_env(ref, kind, amap, N, view):
    ref.harvest.HARVEST_VIEW_SIZE = view
    ref.cleanup.CLEANUP_VIEW_SIZE = view
    cls = ref.HarvestEnv if kind == KIND_HARVEST else ref.CleanupEnv
    env = cls(ascii_map=amap, num_agents=N)
    return env


def gen_actions(rng, cfg, t, steps, N, p_clean, p_fire, p_absent, shuffle_order):
    acts = rng.randint(cfg.num_actions, size=N)
    if p_clean and t < (steps * 3) // 5:
        acts[rng.rand(N) < p_clean] = 8
    if p_fire:
        acts[rng.rand(N) < p_fire] = 7
    absent = rng.rand(N) < p_absent if p_absent else np.zeros(N, bool)
    order = rng.permutation(N) if shuffle_order else np.arange(N)
    return np.where(absent, -1, acts).astype(np.int8), order.astype(np.uint8)


def record(name, kind, amap, N, n_envs, steps, view=7, mode="tape", p_clean=0.0, p_fire=0.0,
           p_absent=0.0, shuffle_order=False, seed0=0, reset_at=(), seeded=False, obs_every=1):
    ref = rh.load_reference()
    cfg = EnvConfig(kind, amap, N, view_size=view)
    B, T, V, H, W = n_envs, steps, cfg.view_width, cfg.height, cfg.width
    nw = len(cfg.waste_points)
    out = dict(kind=kind, ascii_map=np.array(amap), num_agents=N, view_size=view, mode=mode,
               seeds=np.zeros(B, np.uint64), env_ids=np.zeros(B, np.uint64),
               reset_at=np.array(sorted(reset_at), np.int32),
               init_grid=np.zeros((B, H, W), np.uint8), init_pos=np.zeros((B, N, 2), np.int16),
               init_ori=np.zeros((B, N), np.uint8), init_obs=np.zeros((B, N, V, V, 3), np.uint8),
               actions=np.zeros((T, B, N), np.int8), order=np.zeros((T, B, N), np.uint8),
               grid=np.zeros((T, B, H, W), np.uint8), pos=np.zeros((T, B, N, 2), np.int16),
               ori=np.zeros((T, B, N), np.uint8), reward=np.zeros((T, B, N), np.int32),
               obs=np.zeros((T, B, N, V, V, 3), np.uint8), n_draws=np.zeros((T, B), np.int32))
    if reset_at:
        R = len(reset_at)
        out.update(reset_grid=np.zeros((R, B, H, W), np.uint8), reset_pos=np.zeros((R, B, N, 2), np.int16),
                   reset_ori=np.zeros((R, B, N), np.uint8), reset_obs=np.zeros((R, B, N, V, V, 3), np.uint8))
    if mode == "tape":
        out.update(move_order=np.full((T, B, N), 255, np.uint8),
                   waste_order=np.zeros((T, B, nw), np.uint16), waste_shuffled=np.zeros((T, B), np.uint8))
    u_chunks = [[None] * B for _ in range(T)]
    events = dict(waste_spawn_steps=0, apple_prob_steps=0, shared_cell_steps=0, hits=0)

    def store_obs(dst, obs):
        for a in range(N):
            dst[a] = rh.obs_u8(obs['agent-%d' % a])

    for b in range(B):
        seed = seed0 + b
        rng = np.random.RandomState(seed + 4242)
        if mode == "tape":
            np.random.seed(seed)
            random.seed(seed)
            ctx = rh.TapeRecorder()
            out["seeds"][b] = seed
        else:
            pseed = (0x9E3779B97F4A7C15 * (seed + 1)) & 0xFFFFFFFFFFFFFFFF  # exercise both key words
            env_id = 1000003 * b + seed
            ctx = rh.PhiloxIn(pseed)
            out["seeds"][b], out["env_ids"][b] = pseed, env_id
        with ctx:
            if mode == "philox":
                ctx.set(env_id, 0, "reset")
            env = make_env(ref, kind, amap, N, view)
            if mode == "philox":
                ctx.set(env_id, 0, "reset")
            obs = env.reset()
            out["init_grid"][b], out["init_pos"][b], out["init_ori"][b] = rh.extract_state(env)
            store_obs(out["init_obs"][b], obs)
            if seeded:
                st = np.random.get_state()
                assert st[0] == 'MT19937' and st[3] == 0
                out.setdefault("np_state", np.zeros((B, 625), np.uint32))[b] = list(st[1]) + [st[2]]
                ps = random.getstate()
                assert ps[0] == 3 and ps[2] is None
                out.setdefault("py_state", np.zeros((B, 625), np.uint32))[b] = ps[1]
                if nw:
                    out.setdefault("waste_init", np.zeros((B, nw), np.uint16))[b] = [int(r) * W + int(c) for r, c in env.waste_points]
            for t in range(T):
                if t in reset_at:
                    assert mode == "philox"
                    ctx.set(env_id, t, "reset")
                    obs = env.reset()
                    ri = sorted(reset_at).index(t)
                    out["reset_grid"][ri, b], out["reset_pos"][ri, b], out["reset_ori"][ri, b] = rh.extract_state(env)
                    store_obs(out["reset_obs"][ri, b], obs)
                a8, order = gen_actions(rng, cfg, t, T, N, p_clean, p_fire, p_absent, shuffle_order)
                ad = {'agent-%d' % a: int(a8[a]) for a in order if a8[a] >= 0}
                if mode == "tape":
                    obs, rew, dones, info = ctx.step(env, ad)
                    u = list(ctx.uniforms)
                    if ctx.move_order is not None:
                        out["move_order"][t, b, :len(ctx.move_order)] = ctx.move_order
                    if ctx.waste_order is not None:
                        out["waste_shuffled"][t, b] = 1
                        out["waste_order"][t, b] = [r * W + c for r, c in ctx.waste_order]
                    else:  # a valid permutation anyway, so a replay never reads garbage
                        out["waste_order"][t, b] = [int(r) * W + int(c) for r, c in cfg.waste_points]
                    events["waste_spawn_steps"] += ctx.waste_order is not None
                else:
                    ctx.set(env_id, t, "step")
                    obs, rew, dones, info = env.step(ad)
                    u = [0.0] * ctx.k_uniform
                assert dones == dict({'agent-%d' % a: False for a in range(N)}, __all__=False) and info == {}
                out["actions"][t, b], out["order"][t, b] = a8, order
                out["grid"][t, b], out["pos"][t, b], out["ori"][t, b] = rh.extract_state(env)
                out["reward"][t, b] = [rew['agent-%d' % a] for a in range(N)]
                store_obs(out["obs"][t, b], obs)
                out["n_draws"][t, b] = len(u)
                u_chunks[t][b] = u
                events["shared_cell_steps"] += len({tuple(p) for p in out["pos"][t, b].tolist()}) < N
                events["hits"] += int((out["reward"][t, b] <= -50).sum())
                if kind == KIND_CLEANUP:
                    events["apple_prob_steps"] += env.current_apple_spawn_prob > 0
    if mode == "tape":
        out["u_flat"] = np.array([x for t in range(T) for b in range(B) for x in u_chunks[t][b]], np.float64)
    if seeded:  # keep the generator states, drop what they regenerate (after checking that they do)
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import golden_util
        u_re, w_re = golden_util.regenerate_tape(out)
        off = 0
        for t in range(T):
            for b in range(B):
                n = int(out["n_draws"][t, b])
                assert np.array_equal(u_re[t, b, :n], out["u_flat"][off:off + n]), (name, t, b)
                off += n
        sh = out["waste_shuffled"].astype(bool)  # steps without a waste pass recorded the canonical order as a placeholder
        assert np.array_equal(w_re[sh], out["waste_order"][sh]), name
        del out["u_flat"], out["waste_order"]
    if obs_every > 1:
        keep = np.array(sorted(set(range(0, T, obs_every)) | {T - 1}), np.int32)
        out["obs_steps"], out["obs"] = keep, out["obs"][keep]
    path = os.path.join(OUT, name + ".npz")
    with zipfile.ZipFile(path, "w", zipfile.ZIP_LZMA) as zf:
        for k, a in out.items():
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asanyarray(a), allow_pickle=False)
            zf.writestr(k + ".npy", buf.getvalue())
    print("%-28s %7.1f KB  %s" % (name, os.path.getsize(path) / 1024.0, events))


def main():
    tiled = tile_map(CLEANUP_MAP)
    only = sys.argv[1:]
    if only:  # python tests/golden/make_golden.py cleanup_tape64 ...: regenerate the named fixtures only
        global record
        _rec = record
        record = lambda name, *a, **k: _rec(name, *a, **k) if name in only else None
    record("harvest_tape", KIND_HARVEST, HARVEST_MAP, 5, 8, 150, p_fire=0.1)
    record("cleanup_tape", KIND_CLEANUP, CLEANUP_MAP, 5, 8, 250, p_clean=0.4, p_fire=0.05, seeded=True)
    record("cleanup10_tiled_tape", KIND_CLEANUP, tiled, 10, 4, 80, p_clean=0.3, p_fire=0.25, seed0=50, seeded=True)
    record("harvest_dense_tape", KIND_HARVEST, DENSE_MAP, 8, 6, 300, p_absent=0.1, shuffle_order=True, seed0=20)
    record("harvest_r5_tape", KIND_HARVEST, HARVEST_MAP, 5, 2, 40, view=5, p_fire=0.15, seed0=30)
    record("harvest_r10_tape", KIND_HARVEST, HARVEST_MAP, 5, 2, 40, view=10, p_fire=0.15, seed0=32)
    record("cleanup_order_tape", KIND_CLEANUP, CLEANUP_MAP, 5, 4, 120, p_clean=0.4, p_fire=0.1,
           p_absent=0.15, shuffle_order=True, seed0=40)
    # BASELINE.json configs[1] / SURVEY 8d config 2: 64 distinct reference envs x 200 steps (tiled to 4096 slots by the test);
    # CLEAN-biased for the first 120 steps so that the waste density falls below the depletion threshold
    record("cleanup_tape64", KIND_CLEANUP, CLEANUP_MAP, 5, 64, 200, p_clean=0.35, p_fire=0.05, seed0=100, seeded=True, obs_every=5)
    # BASELINE.json configs[3] / SURVEY 8d config 4: 64 reference envs on the 2x2-tiled map, 10 agents, P(FIRE) = P(CLEAN) = 0.25
    record("cleanup10_tiled_tape64", KIND_CLEANUP, tiled, 10, 64, 80, p_clean=0.25, p_fire=0.25, seed0=200, seeded=True, obs_every=8)
    # BASELINE.json configs[2] (the headline workload) under the PRODUCTION random streams: 64 reference envs x 200 steps driven by
    # the Philox streams the kernels draw from, reset() included, one mid-episode reset
    record("harvest_philox64", KIND_HARVEST, HARVEST_MAP, 5, 64, 200, mode="philox", p_fire=0.05, seed0=300, reset_at=(120,), obs_every=10)
    record("harvest_philox", KIND_HARVEST, HARVEST_MAP, 5, 4, 100, mode="philox", p_fire=0.1, reset_at=(50,))
    record("cleanup_philox", KIND_CLEANUP, CLEANUP_MAP, 5, 4, 160, mode="philox", p_clean=0.5, reset_at=(130,))
    record("cleanup10_tiled_philox", KIND_CLEANUP, tiled, 10, 2, 90, mode="philox", p_clean=0.65, p_fire=0.1, seed0=3)


if __name__ == "__main__":
    main()
