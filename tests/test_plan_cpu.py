"""
CPU tests of the MPPI planner's semantics (include/sg_b200.h, sg_plan_sample / sg_plan_update): the numpy noise2
against the oracle's C noise2 bit for bit, and the numpy restatement of sampling and update (tests/plan_oracle.py)
against direct per-element loops written from the header's formulas.
"""
import math

import numpy as np
import pytest

from plan_oracle import noise2_c, noise2_numpy, sample, update


def test_noise2_numpy_matches_c():
    rng = np.random.default_rng(0)
    i = np.concatenate([np.arange(64), 2**40 + np.arange(-32, 32), rng.integers(0, 2**62, 256),
                        [2**63 - 1]]).astype(np.int64)
    for seed in (0, 1, 12345, 2**63 + 17, 2**64 - 1):
        for k in (0, 1, 2, 1000, 2**31 - 1):
            c, py = noise2_c(seed, i, k), noise2_numpy(seed, i, k)
            assert np.array_equal(c.view(np.uint64), py.view(np.uint64)), (seed, k)
    z = noise2_c(3, np.arange(200000), 5)
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1.0) < 0.01  # (a sanity check that it is N(0, 1))


def sample_loop(mu, reset, slots, B, H, seed, k, sigma, dtype):
    N, A = slots.shape
    mu0 = mu.copy()
    table = np.full((N, B, H, A, 2), np.nan)
    for n in range(N):
        for a in range(A):
            if slots[n, a] < 0:
                continue
            if reset is not None and reset[n]:
                mu0[n, :, a] = 0.0
            for b in range(B):
                for h in range(H):
                    z = noise2_c(seed, np.array([((n * A + a) * B + b) * H + h]), k)[0]
                    for c in range(2):
                        eps = sigma[c] * z[c] if b >= 1 else 0.0
                        table[n, b, h, a, c] = dtype(mu0[n, h, a, c] + eps)
    return mu0, table


def update_loop(mu, table, R, lam):
    N, B, H, A, _ = table.shape
    new, shifted = np.zeros_like(mu), np.zeros_like(mu)
    best, rbest = np.zeros((N, A), np.int32), np.zeros((N, A), np.float32)
    for n in range(N):
        for a in range(A):
            rmax = max(float(R[n, b, a]) for b in range(B))
            best[n, a] = min(b for b in range(B) if float(R[n, b, a]) == rmax)
            rbest[n, a] = rmax
            w = [math.exp((float(R[n, b, a]) - rmax) / lam) for b in range(B)]
            for h in range(H):
                for c in range(2):
                    acc = wsum = 0.0
                    for b in range(B):
                        acc += w[b] * (float(table[n, b, h, a, c]) - mu[n, h, a, c])
                        wsum += w[b]
                    new[n, h, a, c] = mu[n, h, a, c] + acc / wsum
    shifted[:, :-1] = new[:, 1:]
    return new, new[:, 0].astype(np.float32), shifted, best, rbest


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_sample_matches_loop(dtype):
    rng = np.random.default_rng(1)
    N, A, B, H = 3, 3, 4, 5
    slots = np.array([[0, 2, -1], [1, -1, -1], [3, 0, 2]], np.int32)
    mu = rng.normal(size=(N, H, A, 2))
    reset = np.array([0, 1, 0], np.uint8)
    sigma = (1.5, 0.2)
    mu0, tab = sample(mu, reset, slots, B, H, 9, 4, sigma, dtype)
    mu0_l, tab_l = sample_loop(mu, reset, slots, B, H, 9, 4, sigma, dtype)
    real = slots >= 0
    assert np.array_equal(mu0.transpose(0, 2, 1, 3)[real], mu0_l.transpose(0, 2, 1, 3)[real])
    assert (mu0[1] == 0).all() and np.array_equal(mu0[0], mu[0])
    got, want = tab.transpose(0, 3, 1, 2, 4)[real], tab_l.transpose(0, 3, 1, 2, 4)[real]
    assert got.dtype == dtype and np.array_equal(got, want)
    assert np.array_equal(tab[:, 0], mu0.astype(dtype))  # branch 0 is the mean
    _, flat = sample(mu, None, slots, B, H, 9, 4, (0.0, 0.0), dtype)
    assert np.array_equal(flat, np.broadcast_to(mu[:, None].astype(dtype), flat.shape))  # sigma 0: B copies


def _check_update(mu, tab, R, lam):
    got, want = update(mu, tab, R, lam), update_loop(mu, tab, R, lam)
    for name, g, w in zip(("mean", "action", "shifted", "best_branch", "best_reward"), got, want):
        if name in ("best_branch", "best_reward"):
            assert np.array_equal(g, w), name
        else:
            np.testing.assert_allclose(g, w, rtol=1e-13, atol=1e-15, err_msg=name)
    return got


def test_update_matches_loop():
    rng = np.random.default_rng(2)
    N, A, B, H = 3, 2, 6, 4
    mu = rng.normal(size=(N, H, A, 2))
    tab = (mu[:, None] + rng.normal(size=(N, B, H, A, 2))).astype(np.float32)
    R = rng.normal(size=(N, B, A)).astype(np.float32)
    R[0, 2, 0] = R[0, 4, 0] = R[0, :, 0].max() + 1.0  # a tie: the smaller branch wins
    new, action, shifted, best, rbest = _check_update(mu, tab, R, 0.7)
    assert best[0, 0] == 2
    assert (shifted[:, -1] == 0).all() and np.array_equal(shifted[:, :-1], new[:, 1:])
    assert np.array_equal(action, new[:, 0].astype(np.float32))


def test_update_limits():
    rng = np.random.default_rng(3)
    N, A, B, H = 2, 2, 5, 3
    mu = rng.normal(size=(N, H, A, 2))
    tab = mu[:, None] + rng.normal(size=(N, B, H, A, 2))
    R = rng.normal(size=(N, B, A)).astype(np.float32)
    # a very small temperature: the mean moves onto the best branch (argmax)
    new, _, _, best, _ = _check_update(mu, tab, R, 1e-9)
    for n in range(N):
        for a in range(A):
            np.testing.assert_allclose(new[n, :, a], tab[n, best[n, a], :, a], rtol=1e-12, atol=1e-12)
    # equal rewards: the plain mean of the branches, best branch 0
    Req = np.full((N, B, A), 0.25, np.float32)
    new, _, _, best, rbest = _check_update(mu, tab, Req, 1.0)
    np.testing.assert_allclose(new, mu + (tab - mu[:, None]).mean(axis=1), rtol=1e-12, atol=1e-14)
    assert (best == 0).all() and (rbest == 0.25).all()
