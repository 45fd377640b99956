"""The headline kernel's exploration test in integers (thrl_device.cuh u32_unit_threshold): a Philox draw x explores when
u32_unit(x) = x * 2^-32 < eps, and the kernel tests x < ceil(eps * 2^32) instead, with the threshold clamped to [0, 2^32].

The CPU test restates both sides in numpy (the oracle's `(double)x * (1.0 / 4294967296.0) < eps`, thrl_oracle.c) and checks
that they agree at every edge epsilon, for the draws on both sides of the threshold.  The GPU test runs qtable_scan_lut2 at
such epsilons against the oracle, bit for bit."""
import math

import numpy as np
import pytest

from th_rl_b200 import abi

TWO32 = 4294967296.0

# epsilons at the edges of the integer test: zero and negative (never explore), the smallest subnormal, around one draw
# step (2^-32), generic values, just below 1 (ceil(eps * 2^32) = 2^32: every draw explores, one past the 32-bit range),
# 1 and above, infinities and NaN
EDGE_EPS = [0.0, -0.0, -1.0, 5e-324, 2.0 ** -33, 2.0 ** -32, math.nextafter(2.0 ** -32, 1.0), 3 * 2.0 ** -33,
            math.nextafter(2.0 ** -32, 0.0), 0.1, 0.5, 0.2 + 2.0 ** -40, 1 - 2.0 ** -33, 1 - 2.0 ** -32,
            math.nextafter(1 - 2.0 ** -32, 0.0), math.nextafter(1 - 2.0 ** -32, 1.0), math.nextafter(1.0, 0.0), 1.0,
            math.nextafter(1.0, 2.0), 2.0, math.inf, -math.inf, math.nan]


def threshold(eps):
    """u32_unit_threshold (thrl_device.cuh), restated."""
    y = eps * TWO32
    if not (y > 0.0):
        return 0
    if y > TWO32 - 1:
        return 1 << 32
    return int(math.ceil(y))


def oracle_explores(x, eps):
    """thrl_oracle.c: u = (double)x * (1.0 / 4294967296.0); u < eps."""
    return bool(np.float64(x) * np.float64(1.0 / TWO32) < np.float64(eps))


def test_integer_threshold_equals_the_f64_test():
    rng = np.random.default_rng(3)
    for eps in EDGE_EPS:
        thr = threshold(eps)
        assert 0 <= thr <= 1 << 32
        xs = {0, 1, 2, (1 << 32) - 2, (1 << 32) - 1}
        xs.update(x for x in range(thr - 3, thr + 3) if 0 <= x < 1 << 32)
        xs.update(int(x) for x in rng.integers(0, 1 << 32, size=64, dtype=np.uint64))
        for x in sorted(xs):
            assert (x < thr) == oracle_explores(x, eps), (eps, x, thr)


def _cfg(T=100):
    base = dict(name="QTable", gamma=0.95, alpha=0.1, eps_end=0.001, epsilon=0.5, eps_step=0.9995, states=100, actions=21,
                action_range=[0.2, 0.4], min_memory=T, capacity=T)
    return {"agents": [dict(base), dict(base)],
            "environment": dict(name="NoisyPriceState", noise_prob=0, a=10, b=1, nplayers=2, max_steps=T),
            "training": dict(print_freq=500, epochs=3)}


@pytest.mark.gpu
def test_lut2_at_edge_epsilons_matches_oracle():
    """Each run holds a pair of edge epsilons for its whole call (eps_end = epsilon, so the decay keeps it): actions, tables,
    counters, epsilon and logs equal the oracle's bit for bit, on the headline kernel."""
    import torch
    from oracle import oracle
    from th_rl_b200 import _lib, engine
    eps = [e for e in EDGE_EPS if math.isfinite(e)]
    pairs = [(a, b) for a in eps for b in eps[::-1]][:64]
    R, E, seed = len(pairs), 4, 77
    cfg = _cfg()
    game = oracle.layout(cfg)
    hp = np.empty((R, 2, 4))
    hp[..., 0], hp[..., 1], hp[..., 3] = 0.1, 0.95, 0.9
    hp[..., 2] = np.array(pairs)
    q0, c0, eps0, p0, *_ = oracle.init(game, R, seed=seed, dtype=np.float32, hp=hp, eps0=abi.eps0_from_config(cfg))
    eps0 = np.ascontiguousarray(np.array(pairs, np.float64).reshape(eps0.shape))
    ref = oracle.scan(game, q0, eps0, p0, E, hp=hp, seed=seed, stats=True, trace=True, n_threads=0)
    b = engine.RunBatch(cfg, R, dtype=torch.float32, seed=seed, hp=hp)
    b.load_state(q0, eps0, p0)
    out = b.scan(E, n_log_runs=R, stats=True, trace=True)
    torch.cuda.synchronize()
    assert _lib.last_kernel() == "lut2", _lib.last_kernel()
    assert np.array_equal(out.trace_actions.cpu().numpy(), ref.trace_actions)
    assert np.array_equal(b.q.cpu().numpy(), ref.q)
    assert np.array_equal(b.counter.cpu().numpy().view(np.uint32), ref.counter)
    assert np.array_equal(b.eps.cpu().numpy(), ref.eps)
    assert np.array_equal(b.price.cpu().numpy(), ref.price)
    assert np.array_equal(out.rewards_log.cpu().numpy(), ref.rewards_log)
    assert np.array_equal(out.stats.cpu().numpy(), ref.stats)
    assert np.array_equal(b.eps.cpu().numpy(), eps0)  # the edge values held for the whole call
