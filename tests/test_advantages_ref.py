"""oracle/advantage_ref.py, the float64 checker of the advantage kernels, pinned without a GPU: a hand-worked trajectory in all
three modes, and plain scipy.signal.lfilter on columns without dones."""
import numpy as np
import scipy.signal

from oracle import advantage_ref as ref

# One env with one agent, T = 4, the episode ends with step 1.  gamma = 0.5, lambda = 0.5 (gamma lambda = 0.25), bootstrap 10.
# The step reward is rewards + 0.5 * intrinsic = [1, 2, 2, 4] + 0.5 * [0, 0, 2, 0] = [1, 2, 3, 4]; values V = [0.5, 1, 1.5, 2].
# Fragments: steps 0-1 with last_r = 0 (done at 1), steps 2-3 with last_r = bootstrap = 10.
REWARDS = np.array([[1], [2], [2], [4]], np.int32)
INTRINSIC = np.array([[0], [0], [2], [0]], np.float32)
VALUES = np.array([[0.5], [1.0], [1.5], [2.0]], np.float32)
DONES = np.array([[0], [1], [0], [0]], np.uint8)
BOOT = np.array([10.0], np.float32)
# log rho = log [1, 2, 0.5, 4]; clip_rho 1: rho_bar = c = [1, 1, 0.5, 1]; clip_pg 2: rho_pg = [1, 2, 0.5, 2]
LOG_RHO = np.log(np.array([[1.0], [2.0], [0.5], [4.0]]))


def test_hand_worked_gae():
    # delta_0 = 1 + 0.5 * 1 - 0.5 = 1        delta_1 = 2 + 0.5 * 0 - 1 = 1       (last_r = 0 after the done)
    # delta_2 = 3 + 0.5 * 2 - 1.5 = 2.5      delta_3 = 4 + 0.5 * 10 - 2 = 7
    # adv_1 = 1, adv_0 = 1 + 0.25 * 1 = 1.25;  adv_3 = 7, adv_2 = 2.5 + 0.25 * 7 = 4.25;  value targets = adv + V
    adv, vt = ref.compute_advantages(REWARDS, VALUES, DONES, BOOT, 0.5, 0.5, True, INTRINSIC, 0.5)
    np.testing.assert_allclose(adv[:, 0], [1.25, 1.0, 4.25, 7.0], rtol=0, atol=1e-12)
    np.testing.assert_allclose(vt[:, 0], [1.75, 2.0, 5.75, 9.0], rtol=0, atol=1e-12)


def test_hand_worked_returns():
    # ret_1 = 2, ret_0 = 1 + 0.5 * 2 = 2;  ret_3 = 4 + 0.5 * 10 = 9, ret_2 = 3 + 0.5 * 9 = 7.5
    adv, vt = ref.compute_advantages(REWARDS, VALUES, DONES, BOOT, 0.5, 0.5, False, INTRINSIC, 0.5)
    np.testing.assert_allclose(adv[:, 0], [2.0, 2.0, 7.5, 9.0], rtol=0, atol=1e-12)
    assert vt is None


def test_hand_worked_vtrace():
    # delta_0 = 1 * (1 + 0.5 * 1 - 0.5) = 1      delta_1 = 1 * (2 + 0 - 1) = 1
    # delta_2 = 0.5 * (3 + 0.5 * 2 - 1.5) = 1.25  delta_3 = 1 * (4 + 0.5 * 10 - 2) = 7
    # vs - V: acc_1 = 1, acc_0 = 1 + 0.5 * 1 * 1 = 1.5;  acc_3 = 7, acc_2 = 1.25 + 0.5 * 0.5 * 7 = 3
    # vs = [2, 2, 4.5, 9];  vs_{t+1} = [2, 0 (done), 9, 10 (bootstrap)]
    # pg_0 = 1 * (1 + 0.5 * 2 - 0.5) = 1.5   pg_1 = 2 * (2 + 0 - 1) = 2   pg_2 = 0.5 * (3 + 0.5 * 9 - 1.5) = 3   pg_3 = 2 * (4 + 5 - 2) = 14
    vs, pg = ref.vtrace(REWARDS, VALUES, DONES, BOOT, LOG_RHO, np.zeros_like(LOG_RHO), 0.5, 1.0, 2.0, INTRINSIC, 0.5)
    np.testing.assert_allclose(vs[:, 0], [2.0, 2.0, 4.5, 9.0], rtol=0, atol=1e-12)
    np.testing.assert_allclose(pg[:, 0], [1.5, 2.0, 3.0, 14.0], rtol=0, atol=1e-12)


def test_bootstrap_behind_a_done_at_the_last_step_is_ignored():
    dones = DONES.copy()
    dones[3] = 1
    for boot in (np.array([np.nan], np.float32), np.array([np.inf], np.float32)):
        adv, vt = ref.compute_advantages(REWARDS, VALUES, dones, boot, 0.5, 0.5, True, INTRINSIC, 0.5)
        ret, _ = ref.compute_advantages(REWARDS, VALUES, dones, boot, 0.5, 0.5, False, INTRINSIC, 0.5)
        vs, pg = ref.vtrace(REWARDS, VALUES, dones, boot, LOG_RHO, np.zeros_like(LOG_RHO), 0.5, 1.0, 2.0, INTRINSIC, 0.5)
        for out in (adv, vt, ret, vs, pg):
            assert np.isfinite(out).all()
        np.testing.assert_allclose(adv[:, 0], [1.25, 1.0, 2.5 + 0.25 * 2.0, 2.0], rtol=0, atol=1e-12)   # delta_3 = 4 - 2


def test_against_plain_lfilter_without_dones():
    rng = np.random.RandomState(0)
    t_count, m, gamma, lam = 50, 6, 0.97, 0.9
    r = rng.randn(t_count, m).astype(np.float32)
    v = rng.randn(t_count, m).astype(np.float32)
    boot = rng.randn(m).astype(np.float32)
    dones = np.zeros((t_count, 3), np.uint8)
    adv, vt = ref.compute_advantages(r, v, dones, boot, gamma, lam, True)
    ret, _ = ref.compute_advantages(r, v, dones, boot, gamma, lam, False)
    for j in range(m):
        vp = np.concatenate([v[:, j], [boot[j]]]).astype(np.float64)
        delta = r[:, j] + gamma * vp[1:] - vp[:-1]
        want = scipy.signal.lfilter([1], [1, -gamma * lam], delta[::-1])[::-1]
        np.testing.assert_allclose(adv[:, j], want, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(vt[:, j], want + v[:, j], rtol=1e-12, atol=1e-12)
        want = scipy.signal.lfilter([1], [1, -gamma], np.concatenate([r[:, j], [boot[j]]]).astype(np.float64)[::-1])[::-1][:-1]
        np.testing.assert_allclose(ret[:, j], want, rtol=1e-12, atol=1e-12)
    # on-policy V-trace with clips >= 1 is GAE with lambda = 1
    zero = np.zeros_like(r)
    vs, pg = ref.vtrace(r, v, dones, boot, zero, zero, gamma, 1.0, np.inf)
    adv1, vt1 = ref.compute_advantages(r, v, dones, boot, gamma, 1.0, True)
    np.testing.assert_allclose(vs, vt1, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(pg, adv1, rtol=1e-12, atol=1e-12)


def test_fragments_split_at_every_done():
    col = np.array([1, 0, 0, 1, 1, 0], bool)
    assert ref.fragments(col, 7.0) == [(0, 1, 0.0), (1, 4, 0.0), (4, 5, 0.0), (5, 6, 7.0)]
    assert ref.fragments(np.array([0, 0, 1], bool), 7.0) == [(0, 3, 0.0)]
