"""The fused policy kernels (csrc/ssd_policy.cu, ssd_policy_head.cu, SURVEY 8f-4) against two independent checkers of the same
layers (models/conv_to_fcnet_v2.py:36-92 on (obs - 128) / 255): oracle/policy_ref.py, a float64 numpy restatement pinned by a
hand-computed vector (tests/test_host_logic.py), and a plain PyTorch fp32 implementation.  The kernels multiply fp16
operands (weights and activations rounded to 11 significant bits), accumulate in fp32 and use tanh.approx in the LSTM, so the
comparison is to a stated tolerance, not bit-exact: measured max abs errors are 2-3e-4 on the trunk features (values O(1))
and below 1e-3 on logits / value / state after three recurrent steps; the asserted bounds are 2e-3 and 5e-3."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TRUNK_TOL = 2e-3    # max abs error of the trunk features (fp16 operand rounding through three layers; features are O(1))
FWD_TOL = 5e-3      # max abs error of logits / value / h / c over three recurrent steps (adds tanh.approx and fp16 h)
ATOL, RTOL = TRUNK_TOL, 0.0


def _reference_features(w, obs):
    x = (obs.to(torch.float32) - 128.0) / 255.0                      # map_env.py:199
    x = x.permute(0, 3, 1, 2)                                         # NHWC -> NCHW
    k = torch.from_numpy(w["conv_w"]).to(obs.device).permute(3, 2, 0, 1)   # [kh, kw, in, out] -> [out, in, kh, kw]
    y = torch.relu(torch.nn.functional.conv2d(x, k, torch.from_numpy(w["conv_b"]).to(obs.device)))
    y = y.permute(0, 2, 3, 1).reshape(obs.shape[0], -1)              # keras Flatten of NHWC
    y = torch.relu(y @ torch.from_numpy(w["fc1_w"]).to(obs.device) + torch.from_numpy(w["fc1_b"]).to(obs.device))
    return torch.relu(y @ torch.from_numpy(w["fc2_w"]).to(obs.device) + torch.from_numpy(w["fc2_b"]).to(obs.device))


@pytest.mark.parametrize("m", [1, 127, 128, 129, 5 * 1024 + 3])
def test_trunk_matches_fp32_reference_random_pixels(m):
    from sequential_social_dilemma_games_b200 import policy
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    w = policy.random_weights(num_outputs=8, seed=3)
    net = policy.ConvToFCNet(w)
    g = torch.Generator(device="cuda").manual_seed(m)
    obs = torch.randint(0, 256, (m, 15, 15, 3), dtype=torch.uint8, device="cuda", generator=g)
    got = net.features(obs)
    want = _reference_features(w, obs)
    torch.cuda.synchronize()
    assert got.shape == (m, 32)
    assert torch.isfinite(got).all()
    err = (got - want).abs().max().item()
    assert err < TRUNK_TOL, "max abs err %g vs torch fp32 (ref max %g)" % (err, want.abs().max().item())
    from oracle import policy_ref
    want64 = policy_ref.features(w, obs.cpu().numpy())           # float64 numpy oracle
    err64 = np.abs(got.cpu().numpy().astype(np.float64) - want64).max()
    assert err64 < TRUNK_TOL, "max abs err %g vs the float64 oracle" % err64
    assert np.abs(want.cpu().numpy() - want64).max() < 1e-4       # the two checkers agree far below the kernel's tolerance
    assert want.abs().max().item() > 0.1   # the comparison is not vacuous


def _reference_forward(w, obs, h, c):
    """conv_to_fcnet_v2.py:68-92 in fp32: Keras LSTM cell (gates i, f, c~, o; sigmoid recurrent activation), linear heads."""
    t = lambda k: torch.from_numpy(w[k]).to(obs.device)
    x = _reference_features(w, obs)
    gates = x @ t("lstm_w") + h @ t("lstm_u") + t("lstm_b")
    i, f, g, o = gates.chunk(4, dim=1)
    c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
    h = torch.sigmoid(o) * torch.tanh(c)
    return h @ t("logits_w") + t("logits_b"), (h @ t("value_w") + t("value_b")).squeeze(1), h, c


def _check_forward_over_steps(cell_size, num_outputs):
    """Three recurrent steps against the fp32 reference and the float64 oracle carried alongside.  cell_size 128 with 1..15
    outputs takes the fused kernel (fp16 operands, tanh.approx) -- 15 outputs put the value in the last of its 16 head columns,
    1 output in column 1 -- and is also run through forward_unfused; every other shape takes the unfused route only (bf16
    GEMM operands around the one-pass cell update)."""
    from sequential_social_dilemma_games_b200 import policy
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    m, u = 1000, cell_size
    fused = cell_size == 128 and num_outputs <= 15
    w = policy.random_weights(num_outputs=num_outputs, cell_size=cell_size, seed=11)
    net = policy.ConvToFCNet(w)
    assert net._fused_head == fused
    g = torch.Generator(device="cuda").manual_seed(5)
    h, c = net.initial_state(m)                                 # tiled layout of the fused kernel, [m, u] rows otherwise
    assert h.shape == ((8, 8, 128, 16) if fused else (m, u))
    hr, cr = torch.zeros((m, u), device="cuda"), torch.zeros((m, u), device="cuda")
    hu, cu = hr.clone(), cr.clone()
    from oracle import policy_ref
    h64, c64 = np.zeros((m, u)), np.zeros((m, u))
    if fused:
        assert torch.equal(net.state_rows(net.state_from_rows(torch.arange(m * 128.0, device="cuda").reshape(m, 128)), m),
                           torch.arange(m * 128.0, device="cuda").reshape(m, 128))
    for _ in range(3):
        obs = torch.randint(0, 256, (m, 15, 15, 3), dtype=torch.uint8, device="cuda", generator=g)
        logits, value, h, c = net.forward(obs, h, c)            # fused tcgen05 LSTM + heads, or the unfused route
        l2, v2, h2, c2 = net.forward_unfused(obs, hu, cu)       # library GEMMs + one-pass cell update
        hu, cu = h2, c2
        lr, vr, hr, cr = _reference_forward(w, obs, hr, cr)
        l64, v64, h64, c64 = policy_ref.forward(w, obs.cpu().numpy(), h64, c64)   # float64 numpy oracle carried alongside
        assert logits.shape == (m, num_outputs) and value.shape == (m,)
        for got, want, w64 in ((logits, lr, l64), (value, vr, v64), (net.state_rows(h, m), hr, h64), (net.state_rows(c, m), cr, c64)):
            assert np.abs(want.cpu().numpy().astype(np.float64) - w64).max() < 2e-4           # torch fp32 vs float64: the checkers agree
            if fused:   # fp16 operands, fp32 accumulation, tanh.approx
                assert (got - want).abs().max().item() < FWD_TOL, (got - want).abs().max().item()
                assert np.abs(got.cpu().numpy().astype(np.float64) - w64).max() < FWD_TOL
            else:       # the unfused route: bf16 operands, 8 significant bits
                assert torch.allclose(got, want, atol=3e-2, rtol=3e-2), (got - want).abs().max().item()
                assert np.allclose(got.cpu().numpy().astype(np.float64), w64, atol=3e-2, rtol=3e-2)
        for got, want in ((l2, lr), (v2, vr), (h2, hr), (c2, cr)):
            assert torch.allclose(got, want, atol=3e-2, rtol=3e-2), (got - want).abs().max().item()   # bf16 operands: 8 significant bits
    assert lr.abs().max().item() > 0.01 and vr.abs().max().item() > 0.01   # not vacuous
    net.close()


def test_forward_matches_fp32_reference_over_steps():
    _check_forward_over_steps(cell_size=128, num_outputs=9)


@pytest.mark.parametrize("cell_size,num_outputs", [(128, 1), (128, 15), (128, 16), (8, 3), (24, 5), (64, 8), (256, 8)])
def test_forward_matches_fp32_reference_every_head_width(cell_size, num_outputs):
    """1 and 15 outputs on the fused head, 16 outputs (the unfused fallback), and cell sizes 8, 24, 64, 256 (unfused)."""
    _check_forward_over_steps(cell_size, num_outputs)


def test_fused_sampling_follows_softmax():
    """`act` samples inside the kernel (Gumbel-max on Philox): frequencies over many agents with IDENTICAL inputs must match
    softmax(logits); a different counter gives different draws, the same (seed, counter) the same ones."""
    from sequential_social_dilemma_games_b200 import policy
    m = 200000
    w = policy.random_weights(num_outputs=8, cell_size=128, seed=2)
    w["logits_w"] = (w["logits_w"] * 4).astype(np.float32)      # spread the probabilities
    net = policy.ConvToFCNet(w)
    one = torch.randint(0, 256, (1, 15, 15, 3), dtype=torch.uint8, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    obs = one.expand(m, 15, 15, 3).contiguous()
    h, c = net.initial_state(m)
    net.seed_sampling(77)
    a1, value, h1, c1 = net.act(obs, h, c)
    a2, _, _, _ = net.act(obs, h, c)
    net.seed_sampling(77)
    a3, _, _, _ = net.act(obs, h, c)
    logits = net.forward(obs[:1], *net.initial_state(1))[0][0]
    p = torch.softmax(logits.double(), 0).cpu().numpy()
    assert a1.dtype == torch.int8 and int(a1.min()) >= 0 and int(a1.max()) < 8
    freq = np.bincount(a1.cpu().numpy().astype(np.int64), minlength=8) / m
    assert np.abs(freq - p).max() < 5 * np.sqrt(p.max() / m) + 1e-3, (freq, p)   # five sigma of a binomial frequency
    assert torch.equal(a1, a3) and not torch.equal(a1, a2)
    net.close()


def test_trunk_on_env_observations_and_rollout_loop():
    """Observations straight from the step kernel; a short closed loop env -> policy -> env with no host round trip."""
    from sequential_social_dilemma_games_b200 import policy
    from sequential_social_dilemma_games_b200.batched import BatchedSSDEnv, make_config
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    env = BatchedSSDEnv(make_config("harvest", num_agents=5), 300, seed=5)
    w = policy.random_weights(num_outputs=8, seed=1)
    net = policy.ConvToFCNet(w)
    obs = env.reset()
    h, c = net.initial_state(300 * 5)
    gen = torch.Generator(device="cuda").manual_seed(0)
    for _ in range(6):
        flat = obs.reshape(-1, 15, 15, 3)
        got = net.features(flat)
        want = _reference_features(w, flat)
        assert (got - want).abs().max().item() < TRUNK_TOL, (got - want).abs().max().item()
        a, value, h, c = net.act(flat, h, c, generator=gen)
        assert a.dtype == torch.int8 and int(a.min()) >= 0 and int(a.max()) < 8
        obs, rew = env.step(a.reshape(300, 5))
    torch.cuda.synchronize()
    env.close()
    net.close()
