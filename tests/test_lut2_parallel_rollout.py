"""The headline kernel's lane-parallel rollout (qtable_scan_lut2 phase B, DESIGN.md 4.1).  An episode with few exploration
steps ("events") is played from the powers of the greedy successor function, 32 steps per pass; others step by step.

Replayed draws (THRL_RNG_REPLAY_DRAWS) place every event exactly: an agent explores at step t when its draw is below its
epsilon (held at 0.5 here), with the replayed action as the forced one.  Each case is compared with the oracle bit for bit:
per-step actions, rewards and prices, tables, counters, epsilon, the outgoing price, logs and statistics.  Which rollout a
case takes follows from the restated plan (`parallel_rollout` below); the CPU test pins every case to the path it is named
for, so that a change of the threshold or of the plan cannot quietly move a case to the other side."""
import os
import sys

import numpy as np
import pytest

from th_rl_b200 import abi

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_lut2_plan_edges import lut2_plan  # noqa: E402

MAX_EVENTS = 12  # kLut2MaxEvents (thrl_scan_lut2.cuh)


def parallel_rollout(NS, T, n_events):
    """The noise-free kernel plays an episode lane-parallel when it fits the plan: T <= 128, NS + 1 <= 64 states, at most
    kLut2MaxEvents steps in which an agent explores."""
    return 0 < T <= 128 and NS + 1 <= 64 and n_events <= MAX_EVENTS


def _cfg(T, states=100, actions=21):
    base = dict(name="QTable", gamma=0.95, alpha=0.1, eps_end=0.5, epsilon=0.5, eps_step=0.9, states=states,
                actions=actions, action_range=[0.2, 0.4], min_memory=T, capacity=T)
    return {"agents": [dict(base), dict(base)],
            "environment": dict(name="NoisyPriceState", noise_prob=0, a=10, b=1, nplayers=2, max_steps=T),
            "training": dict(print_freq=500, epochs=3)}


# grids: (T, states, actions); NS = 41 for 100 x 21, 63 for 200 x 32 and 64 for 285 x 31
GRIDS = {
    "T100": (100, 100, 21),
    "T1": (1, 100, 21),
    "T33": (33, 100, 21),
    "T127": (127, 100, 21),
    "T128": (128, 100, 21),
    "T129": (129, 100, 21),
    "NS63": (100, 200, 32),
    "NS64": (100, 285, 31),
}
GRID_NS = {"T100": 41, "T1": 41, "T33": 41, "T127": 41, "T128": 41, "T129": 41, "NS63": 63, "NS64": 64}


def _spread(T, n, first=0):
    """n event steps spread over [first, T)."""
    return sorted({first + (i * (T - first)) // n for i in range(n)}) if n else []


def _schedules(T):
    """name -> [(step, agent mask: 1 = agent 0, 2 = agent 1, 3 = both)], the same in every epoch of a run"""
    s = {
        "none": [],
        "step0": [(0, 3)],
        "last": [(T - 1, 3)],
        "back_to_back": [(t, m) for t, m in [(2, 3), (3, 1), (4, 2), (T - 2, 3), (T - 1, 1)] if 0 <= t < T],
        "agent0_only": [(t, 1) for t in _spread(T, 5, 1)],
        "agent1_only": [(t, 2) for t in _spread(T, 5, 1)],
        "chunk_edges": [(t, m) for t, m in [(31, 3), (32, 1), (63, 2), (64, 3), (95, 1), (96, 2), (127, 3), (128, 1)]
                        if t < T],
        "max_events": [(t, 1 + t % 3) for t in _spread(T, MAX_EVENTS)],
        "max_events_plus_1": [(t, 1 + t % 3) for t in _spread(T, MAX_EVENTS + 1)],
        "32_events": [(t, 3) for t in _spread(T, 32)],
        "33_events": [(t, 3) for t in _spread(T, 33)],
    }
    rng = np.random.default_rng(T)
    s["random"] = [(int(t), int(rng.integers(1, 4))) for t in np.sort(rng.choice(T, size=min(T, 6), replace=False))]
    return {name: [(t, m) for t, m in sch if t < T] for name, sch in s.items()}


def _draws(T, R, E, scheds, A, seed):
    """replay_u (R, E, T, 2): 0 where the agent explores, 1 elsewhere; replay_ra: forced actions"""
    u = np.ones((R, E, T, 2))
    for r, sch in enumerate(scheds):
        for t, m in sch:
            if m & 1:
                u[r, :, t, 0] = 0.0
            if m & 2:
                u[r, :, t, 1] = 0.0
    ra = np.random.default_rng(seed).integers(0, A, size=(R, E, T, 2)).astype(np.int32)
    return u, ra


def test_cases_cover_both_rollouts():
    for name, (T, states, actions) in GRIDS.items():
        plan = lut2_plan(_cfg(T, states, actions), 4, False)
        assert plan.get("NS") == GRID_NS[name], (name, plan)
        assert "rejected" not in plan, (name, plan)
        for case, sch in _schedules(T).items():
            n = len({t for t, _ in sch})
            assert all(0 <= t < T for t, _ in sch), (name, case)
            par = parallel_rollout(plan["NS"], T, n)
            if name in ("T129", "NS64"):
                assert not par, (name, case)
            elif case in ("none", "step0", "last", "back_to_back", "agent0_only", "agent1_only", "random"):
                assert par, (name, case)
            elif case == "max_events" and T >= MAX_EVENTS:
                assert n == MAX_EVENTS and par, (name, case)
            elif case in ("max_events_plus_1", "32_events", "33_events") and T > 33:
                assert not par, (name, case)
    assert parallel_rollout(63, 128, MAX_EVENTS) and not parallel_rollout(64, 128, 0)
    assert not parallel_rollout(41, 129, 0) and not parallel_rollout(41, 100, MAX_EVENTS + 1)


def _run(cfg, scheds, E, u, ra, seed=5):
    import torch
    from oracle import oracle
    from th_rl_b200 import _lib, engine
    R = len(scheds)
    game = oracle.layout(cfg)
    hp = np.empty((R, 2, 4))
    hp[..., 0], hp[..., 1], hp[..., 2], hp[..., 3] = 0.1, 0.95, 0.5, 0.9
    q0, c0, eps0, p0, *_ = oracle.init(game, R, seed=seed, dtype=np.float32, hp=hp, eps0=[0.5, 0.5])
    eps0 = np.full_like(eps0, 0.5)
    ref = oracle.scan(game, q0, eps0, p0, E, hp=hp, rng_mode=abi.THRL_RNG_REPLAY_DRAWS, replay_u=u, replay_ra=ra,
                      stats=True, trace=True, n_threads=0)
    b = engine.RunBatch(cfg, R, dtype=torch.float32, seed=seed, hp=hp)
    b.load_state(q0, eps0, p0)
    out = b.scan(E, rng_mode=abi.THRL_RNG_REPLAY_DRAWS, replay_u=u, replay_ra=ra, n_log_runs=R, stats=True, trace=True)
    torch.cuda.synchronize()
    assert _lib.last_kernel() == "lut2", _lib.last_kernel()
    acts = out.trace_actions.cpu().numpy()
    for r in range(R):
        assert np.array_equal(acts[r], ref.trace_actions[r]), r
    assert np.array_equal(out.trace_rewards.cpu().numpy(), ref.trace_rewards)
    assert np.array_equal(out.trace_prices.cpu().numpy(), ref.trace_prices)
    assert np.array_equal(b.q.cpu().numpy(), ref.q)
    assert np.array_equal(b.counter.cpu().numpy().view(np.uint32), ref.counter)
    assert np.array_equal(b.eps.cpu().numpy(), ref.eps)
    assert np.array_equal(b.price.cpu().numpy(), ref.price)
    assert np.array_equal(out.rewards_log.cpu().numpy(), ref.rewards_log)
    assert np.array_equal(out.actions_log.cpu().numpy(), ref.actions_log)
    assert np.array_equal(out.stats.cpu().numpy(), ref.stats)
    return ref


@pytest.mark.gpu
@pytest.mark.parametrize("grid", sorted(GRIDS))
def test_parallel_rollout_matches_oracle(grid):
    """Every schedule, three epochs (the first starts from the call's initial price, state NS), bit for bit."""
    T, states, actions = GRIDS[grid]
    cfg = _cfg(T, states, actions)
    sch = _schedules(T)
    names = sorted(sch)
    scheds = [sch[n] for n in names]
    u, ra = _draws(T, len(scheds), 3, scheds, actions, seed=T + states)
    _run(cfg, scheds, 3, u, ra)


@pytest.mark.gpu
def test_forced_action_equal_to_the_greedy_one():
    """Events whose forced actions are the greedy ones: the episode is the greedy one, but the steps still count as
    events.  The greedy actions are the oracle's trace of the same epoch without events."""
    T, states, actions = GRIDS["T100"]
    cfg = _cfg(T, states, actions)
    steps = [0, 1, 17, 31, 32, 50, 99]
    R = 4
    u0, ra = _draws(T, R, 1, [[]] * R, actions, seed=9)
    ref = _run(cfg, [[]] * R, 1, u0, ra)
    greedy = ref.trace_actions.reshape(R, 1, T, 2)
    scheds = [[(t, 3) for t in steps], [(t, 1) for t in steps], [(t, 2) for t in steps], [(0, 3), (99, 3)]]
    u, _ = _draws(T, R, 1, scheds, actions, seed=9)
    ra = np.ascontiguousarray(greedy.astype(np.int32))
    ref2 = _run(cfg, scheds, 1, u, ra)
    assert np.array_equal(ref2.trace_actions, ref.trace_actions)  # the same episode as without events
