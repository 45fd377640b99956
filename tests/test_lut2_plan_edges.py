"""The headline kernel (qtable_scan_lut2, thrl_scan_lut2.cuh) at the limits of its plan (plan_lut2, thrl.cu).

`lut2_plan` restates plan_lut2 in Python (as conftest.uses_lattice_kernel restates plan_pwl), and `lpc_fits` the layout
of launch_lpc_gl.  The CPU tests pin every case below to the band it is named for, so that a change to a config or to the
plan cannot silently move a case back into the region the other tests already cover.  The GPU tests play each case on
the kernel and compare everything with the oracle bit for bit: per-step traces, tables, counters, epsilon, price, logs
and statistics.

Cases: compact rows past 64 (phase E's "rescan all" path), up to the plan's limit of 253, and one past it; byte-sized
action indices >= 128 in the packed action word; the joint-action limit; episodes of 1 step, of one and two full update
chunks and the longest the plan takes; full CTAs whose warps play several runs in turn; initial prices whose rows are
staged in the two extra slots (and the aliasing of the two); tables full of ties; chains of transitions that bootstrap
from the row the previous one wrote.
"""
import numpy as np
import pytest

from th_rl_b200 import abi

SMEM_OPTIN_B200 = 232448  # cudaDevAttrMaxSharedMemoryPerBlockOptin of a B200 (227 KB)

# thrl_scan_lut2.cuh / thrl_scan_lpc.cuh constants
MAX_JOINT, MAX_STATES, MAX_ROWS = 1024, 254, 253
MAX_WARPS = {4: 24, 8: 16}
NOISE_WARPS = 16
CHUNK = 16
LPC_MAX_WARPS = 16


def _align(x, a=16):
    return (x + a - 1) // a * a


def _scale(k, A, lo, hi):
    d = float(k) / (float(A) - 1.0)
    d = d * (hi - lo)
    return d + lo


def act_row(price, max_state, states):
    """agents.py:47-49 as the kernel acts on it: float32 price / max_state * states, rounded half to even."""
    x = np.float32(np.float32(price) / np.float32(max_state))
    x = np.float32(x * np.float32(states))
    return int(np.rint(x))


def upd_row(price, max_state, states):
    """The same encode in f64, as the update uses it."""
    return int(np.rint(price / max_state * float(states)))


def joint_prices(game):
    """Price after every joint action (k0 * A1 + k1), with the reference's operation order."""
    A0, A1 = game.agent[0].actions, game.agent[1].actions
    ab = game.a / game.b
    out = []
    for j in range(A0 * A1):
        k0, k1 = j // A1, j % A1
        aq0 = ab * _scale(k0, A0, game.agent[0].action_lo, game.agent[0].action_hi)
        aq1 = ab * _scale(k1, A1, game.agent[1].action_lo, game.agent[1].action_hi)
        pn = game.a - game.b * ((0.0 + aq0) + aq1)
        out.append(pn if pn > 0.0 else (pn if pn != pn else 0.0))
    return out


def encodes(game, price):
    """(act row 0, update row 0, act row 1, update row 1) of a price."""
    s0, s1 = game.agent[0], game.agent[1]
    return (act_row(price, s0.max_state, s0.states), upd_row(price, s0.max_state, s0.states),
            act_row(price, s1.max_state, s1.states), upd_row(price, s1.max_state, s1.states))


def lut2_plan(cfg, elem, noisy, smem_optin=SMEM_OPTIN_B200):
    """plan_lut2 (thrl.cu) restated: a dict with NS, NR[2], L[2], warps (runs per CTA as planned, before launch_lut2 shrinks
    the CTA for small batches) and the compact row lists; or, when the plan rejects the game, {"rejected": reason} with
    whatever was counted before the rejection."""
    from oracle import oracle
    G = oracle.layout(cfg)
    if G.n_agents != 2 or not G.regular:
        return dict(rejected="game")
    A0, A1, T = G.agent[0].actions, G.agent[1].actions, G.max_steps
    if A0 > 255 or A1 > 255 or A0 * A1 > MAX_JOINT or T > 32767:
        return dict(rejected="actions" if T <= 32767 else "T")
    rmax = [0, 0]
    if noisy:
        if not (G.a > 0.0) or not (G.b > 0.0) or T > 200:
            return dict(rejected="noisy T" if T > 200 else "noisy demand")
        lo_sum = 0.0
        for a in range(2):
            lo = min(G.agent[a].action_lo, G.agent[a].action_hi)
            if not (lo >= 0.0):
                return dict(rejected="noisy demand")
            lo_sum += lo
        pmax = G.a - G.a * lo_sum
        if not (pmax >= 0.0):
            pmax = 0.0
        for a in range(2):
            r = pmax / G.agent[a].max_state * float(G.agent[a].states) + 2.5
            rmax[a] = int(r) if r < float(G.agent[a].states) else G.agent[a].states
    tuples = {}
    for price in joint_prices(G):
        if price != price:
            return dict(rejected="price")
        tuples.setdefault(encodes(G, price), len(tuples))
    NS = len(tuples)
    if NS > MAX_STATES:
        return dict(rejected="states", NS=NS)
    rows = [set(), set()]
    for t in tuples:
        rows[0].update((t[0], t[1]))
        rows[1].update((t[2], t[3]))
    if noisy:
        if NS + 1 + T > 255:
            return dict(rejected="noisy state ids", NS=NS)
        for a in range(2):
            if rows[a] and max(rows[a]) > rmax[a]:
                return dict(rejected="noisy rows", NS=NS)
            rows[a].update(range(rmax[a] + 1))
    NR, L = [0, 0], [0, 0]
    for a in range(2):
        if len(rows[a]) > MAX_ROWS or any(r < 0 or r > G.agent[a].states for r in rows[a]):
            return dict(rejected="rows", NS=NS, NR=[len(rows[0]), len(rows[1])])
        NR[a] = len(rows[a])
        s = G.agent[a]
        L[a] = 0 if s.min_memory > s.capacity else min(T, s.capacity)
    J = A0 * A1
    cta = _align(2 * J) + _align(2 * (NR[0] + NR[1])) + J * 32 + _align(J * 8) + _align((A0 + A1) * 8)
    o = _align((NR[0] + 2) * A0 * elem) + _align((NR[1] + 2) * A1 * elem) + _align(NR[0] + NR[1] + 4)
    o += _align((NS + 1 + (T if noisy else 0)) * 4)
    o += max(_align((NS + 2) * 4), CHUNK * 8 + 16)
    if noisy:
        o += _align(T) + _align(T * 8) + _align(T + 1)
    o += _align(2 * T) + max(_align(T * 8), _align(2 * T * elem))
    w = (smem_optin - cta) // o
    if w < 2:
        return dict(rejected="shared memory", NS=NS, NR=NR, L=L)
    wmax = NOISE_WARPS if noisy else MAX_WARPS[elem]
    return dict(NS=NS, NR=NR, L=L, warps=min(w, wmax), rows=[sorted(rows[0]), sorted(rows[1])], warp_bytes=o, cta_bytes=cta)


def lpc_fits(cfg, elem, GL, smem_optin=SMEM_OPTIN_B200):
    """launch_lpc_gl (thrl.cu) restated: does one warp group of the lane-per-chain kernel fit next to its CTA tables?
    Only asked of games the lut2 plan takes noise-free (the kernel reuses that plan)."""
    from oracle import oracle
    plan = lut2_plan(cfg, elem, False, smem_optin)
    assert "rejected" not in plan, plan
    G = oracle.layout(cfg)
    T, NS, NR, L = G.max_steps, plan["NS"], plan["NR"], plan["L"]
    J = G.agent[0].actions * G.agent[1].actions
    cells = max((NR[a] + 2) * G.agent[a].actions for a in range(2))
    rows_max = max(NR[a] + 2 for a in range(2))
    o = _align(cells * GL * elem) + _align(max(1, *L) * GL * elem) + _align(T * GL * 4) + _align(T * GL)
    o += _align((NS + 1) * GL * 4) + _align((NS + 1) * GL * 2) + _align(rows_max * GL) + _align(GL * 8) + _align(2 * GL * 2)
    cta = _align(2 * J) + _align(2 * (NR[0] + NR[1])) + J * 32 + J * 16
    return (smem_optin - cta) // o >= 1


def planned(plan):
    return "rejected" not in plan


# ------------------------------------------------------------------------------------------------ the cases
def _two(T, a0, a1, noise=0.0):
    from test_gpu_parity import _two_agent_cfg
    return _two_agent_cfg(T, a0, a1, env=dict(noise_prob=noise))


def _grid32(states, T=40):
    """32 x 32 actions over slightly different ranges: the prices of the 1024 joint actions spread over many rows."""
    return _two(T, dict(actions=32, states=states, action_range=[0.1, 0.3], min_memory=T),
                dict(actions=32, states=states, action_range=[0.11, 0.29], min_memory=T))


def _c2(T, noise=0.0, actions=(21, 21)):
    """The C2 grid (21 x 21 actions, 100 states), one batch of the whole episode per agent."""
    return _two(T, dict(actions=actions[0], min_memory=T, capacity=T), dict(actions=actions[1], min_memory=T, capacity=T), noise=noise)


def _noisy(cfg):
    return cfg["environment"]["noise_prob"] > 0


T_MAX = 9900  # the longest episode the f32 plan takes on the C2 grid at the B200's opt-in shared memory

# name -> (config, check of the restated f32 and f64 plans: the band the case is named for)
CASES = {
    # compact rows past 64: phase E rescans them all; one pass of the warp over rows 64 .. NR+1
    "rows69": (_grid32(180), lambda p4, p8: all(64 < p["NR"][a] <= 94 for p in (p4, p8) for a in (0, 1))),
    # NR + 2 > 96: two passes; compact indices past 64 in the masks, the snapshot and the update
    "rows113": (_grid32(300), lambda p4, p8: all(94 < p["NR"][a] <= 125 for p in (p4, p8) for a in (0, 1))),
    # kLut2MaxRows: compact indices up to 254 with the initial slots, bytes past 127; f64 tables do not fit twice
    "rows253": (_grid32(724), lambda p4, p8: p4["NR"] == [253, 253] and p4["warps"] == 2 and p8["rejected"] == "shared memory"),
    # one row past the limit: the plan falls back
    "rows254": (_grid32(731), lambda p4, p8: p4["rejected"] == p8["rejected"] == "rows" and max(p4["NR"]) == 254),
    # k0 >= 128 in the packed action word, eight column passes per row
    "a255": (_two(40, dict(actions=255, min_memory=40), dict(actions=4, min_memory=40)), lambda p4, p8: p4["warps"] == 4 and planned(p8)),
    # J = 1024 exactly, on the <= 32-column instantiation
    "a32x32": (_two(40, dict(actions=32, min_memory=40), dict(actions=32, min_memory=40)), lambda p4, p8: planned(p4) and planned(p8)),
    # the first width past 32 columns (row_argmax), J = 1023
    "a33x31": (_two(40, dict(actions=33, min_memory=40), dict(actions=31, min_memory=40)), lambda p4, p8: planned(p4) and planned(p8)),
    # one joint action past the limit
    "J1025": (_two(40, dict(actions=41, min_memory=40), dict(actions=25, min_memory=40)),
              lambda p4, p8: p4["rejected"] == p8["rejected"] == "actions"),
    # 63 update chunks, 32 lane passes of the draws
    "T1000": (_c2(1000), lambda p4, p8: p4["L"] == [1000, 1000] and p4["warps"] == 12 and planned(p8)),
    # the longest episode: two runs per CTA; one step more does not fit
    "Tmax": (_c2(T_MAX), lambda p4, p8: p4["warps"] == 2 and p8["rejected"] == "shared memory"),
    "Tmax_plus1": (_c2(T_MAX + 1), lambda p4, p8: p4["rejected"] == "shared memory"),
    # noisy instantiation: the longest episode it takes, byte-sized state ids at their limit (NS + 1 + T = 255) and one past
    "noisy_T200": (_c2(200, noise=0.6), lambda p4, p8: planned(p4) and planned(p8)),
    "noisy_ids255": (_c2(199, noise=0.6, actions=(33, 31)), lambda p4, p8: p4["NS"] + 1 + 199 == 255 and planned(p8)),
    "noisy_ids256": (_c2(200, noise=0.6, actions=(33, 31)), lambda p4, p8: p4["rejected"] == "noisy state ids" and p4["NS"] + 1 + 200 == 256),
    "noisy_T201": (_c2(201, noise=0.6), lambda p4, p8: p4["rejected"] == p8["rejected"] == "noisy T"),
}
CHUNKED = ("rows113", "rows253", "T1000")
TOO_LONG_FOR_GENERIC = ("Tmax", "Tmax_plus1")

# the cases of test_gpu_parity.test_two_agent_edge_shapes_match_oracle added for these limits (every kernel choice there:
# the lane-per-chain layout must fit in both dtypes and both group widths)
SHORT_CASES = {"T1": [1, 1], "T2": [2, 2], "L16": [16, 16], "L17": [17, 17], "L32": [32, 32]}


@pytest.mark.parametrize("case", sorted(CASES))
def test_case_lies_in_its_band(case):
    cfg, band = CASES[case]
    p4, p8 = lut2_plan(cfg, 4, _noisy(cfg)), lut2_plan(cfg, 8, _noisy(cfg))
    assert band(p4, p8), (p4, p8)


@pytest.mark.parametrize("case", sorted(SHORT_CASES))
def test_short_case_lies_in_its_band(case):
    from test_gpu_parity import TWO_AGENT_CASES
    cfg = TWO_AGENT_CASES[case]
    for elem in (4, 8):
        p = lut2_plan(cfg, elem, False)
        assert p["L"] == SHORT_CASES[case], p
        assert lpc_fits(cfg, elem, 8) and lpc_fits(cfg, elem, 16)


def test_plan_restatement_matches_design_figures():
    """The figures DESIGN.md states for the C2 shape on a B200: 24 runs per SM with f32 tables (8,688 B per run), about 12
    with f64 tables (thrl_scan_lut2.cuh), 15 with demand noise (C2n)."""
    from conftest import load_golden
    cfg = load_golden("c1_example_2q_seed0")["config"]
    p = lut2_plan(cfg, 4, False)
    assert (p["NS"], p["NR"], p["warps"], p["warp_bytes"]) == (41, [41, 41], 24, 8688)
    assert lut2_plan(cfg, 8, False)["warps"] == 12
    cfg["environment"]["noise_prob"] = 0.05
    assert lut2_plan(cfg, 4, True)["warps"] == 15


# ------------------------------------------------------------------------------------------------ initial-price slots
# A grid whose compact rows have gaps (9 x 7 actions over 300 states), so that a price's act row (f32 encode) and update
# row (f64 encode) can each be a compact row or not.  The kernel stages the rows that are not in the two extra slots of
# the agent and aliases the second to the first when the two encodes agree.
GAPS = _two(40, dict(actions=9, states=300, action_range=[0.1, 0.3], min_memory=40),
            dict(actions=7, states=300, action_range=[0.11, 0.29], min_memory=40))
INIT_KINDS = ("both compact", "act compact", "update compact", "neither", "neither, aliased")


def _init_kind(game, rows, a, price):
    s = game.agent[a]
    ta, tu = act_row(price, s.max_state, s.states), upd_row(price, s.max_state, s.states)
    ca, cu = ta in rows, tu in rows
    if ca and cu:
        return "both compact"
    if ca or cu:
        return "act compact" if ca else "update compact"
    return "neither" if ta != tu else "neither, aliased"


def initial_prices(cfg, per_kind=4):
    """Initial prices that give every agent every kind of initial rows at least per_kind times, plus 0 and a (row = states).
    The two encodes disagree only within float32 rounding of a half-row boundary (k + 1/2) * max_state / states."""
    from oracle import oracle
    G = oracle.layout(cfg)
    rows = [set(r) for r in lut2_plan(cfg, 4, False)["rows"]]
    found = {(a, k): [] for a in (0, 1) for k in INIT_KINDS}
    ms, st = G.agent[0].max_state, G.agent[0].states
    assert (ms, st) == (G.agent[1].max_state, G.agent[1].states)
    for k in range(st):
        for d in range(-60, 61):
            x = (k + 0.5) * ms / st * (1.0 + d * 1e-8)
            for a in (0, 1):
                lst = found[(a, _init_kind(G, rows[a], a, x))]
                if len(lst) < per_kind and (not lst or abs(lst[-1] - x) > 0.2):  # spread over the price range
                    lst.append(x)
    prices = sorted({x for v in found.values() for x in v} | {0.0, G.a})
    return np.array(prices), found


def test_initial_prices_reach_every_kind():
    from oracle import oracle
    noisy = _two(40, GAPS["agents"][0], GAPS["agents"][1], noise=0.05)
    assert all(planned(lut2_plan(cfg, elem, _noisy(cfg))) for cfg in (GAPS, noisy) for elem in (4, 8))
    prices, found = initial_prices(GAPS)
    for key, v in found.items():
        assert len(v) >= 3, key
    G = oracle.layout(GAPS)
    assert encodes(G, 0.0) == (0, 0, 0, 0) and encodes(G, G.a) == (300, 300, 300, 300)


# ------------------------------------------------------------------------------------------------ ties and chains
def _hp_grid(R, values, seed):
    """[R, 2, 4] hyper-parameters (alpha, gamma, eps_end, eps_step) with every combination of values = (alphas, gammas,
    epsilons) for agent 0 in turn and a shuffled one for agent 1; epsilon is held (eps_end = epsilon)."""
    import itertools
    combos = list(itertools.product(*values))
    rng = np.random.default_rng(seed)
    hp = np.empty((R, 2, 4))
    for r in range(R):
        for a, c in enumerate((combos[r % len(combos)], combos[rng.integers(len(combos))])):
            hp[r, a] = (c[0], c[1], c[2], 0.9)
    return hp


def tied_state(cfg, R, dtype, seed):
    """Library initial tables rounded to integers (about 7 levels per row, so rows hold equal maxima) with a fifth of the
    rows set to a mix of 0.0 and -0.0; per-run alpha in {0, 0.5, 1}, gamma in {0, 0.99}, epsilon in {0, 0.5} held.  At
    alpha = 0 the tables never change and every greedy choice of the call is a tie-break."""
    from oracle import oracle
    G = oracle.layout(cfg)
    hp = _hp_grid(R, ([0.0, 0.5, 1.0], [0.0, 0.99], [0.0, 0.5]), seed)
    q0, c0, eps0, p0 = oracle.init(G, R, seed=seed, dtype=dtype, hp=hp)
    rng = np.random.default_rng(seed)
    for a in (0, 1):
        t = abi.table_view(q0, G.agent[a])
        assert np.shares_memory(t, q0)
        t[...] = np.round(t)
        zero = rng.random(t.shape[:2]) < 0.2
        t[zero] = rng.choice(np.array([0.0, -0.0], dtype), size=(int(zero.sum()), t.shape[2]))
    return hp, (q0, np.ascontiguousarray(hp[:, :, 2]), p0)


def chain_state(cfg, R, dtype, seed, period):
    """epsilon = 0 (greedy play only).  period 1: zero tables, alpha = 1: both agents play action 0 forever, so from step 1
    on every transition bootstraps from the row it and its predecessor just wrote.  period 2: per run, two joint actions whose
    prices lead to distinct rows; each state's greedy pair (a cell far above the others) leads to the other state, so every
    transition bootstraps from the row its predecessor but one wrote."""
    from oracle import oracle
    G = oracle.layout(cfg)
    hp = np.empty((R, 2, 4))
    hp[..., 0] = 1.0 if period == 1 else np.repeat(np.array([0.1, 0.5, 1.0])[np.arange(R) % 3][:, None], 2, axis=1)
    hp[..., 1], hp[..., 2], hp[..., 3] = 0.95, 0.0, 0.9
    q0, c0, eps0, p0 = oracle.init(G, R, seed=seed, dtype=dtype, hp=hp)
    q0[...] = 0.0
    if period == 2:
        A1 = G.agent[1].actions
        prices = joint_prices(G)
        rng = np.random.default_rng(seed)
        tabs = [abi.table_view(q0, G.agent[a]) for a in (0, 1)]
        for r in range(R):
            while True:
                ja, jb = rng.integers(len(prices), size=2)
                ea, eb = encodes(G, prices[ja]), encodes(G, prices[jb])
                if ea[0] == ea[1] and eb[0] == eb[1] and ea[2] == ea[3] and eb[2] == eb[3] and ea[0] != eb[0] and ea[2] != eb[2]:
                    break
            tabs[0][r, ea[0], jb // A1] = tabs[0][r, eb[0], ja // A1] = 1e4
            tabs[1][r, ea[2], jb % A1] = tabs[1][r, eb[2], ja % A1] = 1e4
            p0[r] = prices[ja]
    return hp, (q0, np.zeros((R, 2)), p0)


def chain_counts(game, p0, trace_prices):
    """Per agent: transitions j whose next update row cn(j) equals cu(j) and cu(j-1) (period 1), and those with
    cn(j) == cu(j-1) != cu(j) (period 2), from the prices of a trace [R, E, T]."""
    R = trace_prices.shape[0]
    after = trace_prices.reshape(R, -1)
    before = np.concatenate([np.asarray(p0).reshape(R, 1), after[:, :-1]], axis=1)
    out = []
    for a in (0, 1):
        s = game.agent[a]
        enc = np.vectorize(lambda x: upd_row(x, s.max_state, s.states))
        cu, cn = enc(before), enc(after)
        p1 = (cn[:, 1:] == cu[:, 1:]) & (cu[:, 1:] == cu[:, :-1])
        p2 = (cn[:, 1:] == cu[:, :-1]) & (cn[:, 1:] != cu[:, 1:])
        out.append((int(p1.sum()), int(p2.sum()), p1.size))
    return out


@pytest.mark.parametrize("period", [1, 2])
def test_chain_premise_holds(period):
    """What the chain cases stand for, read from the oracle's own trace."""
    from oracle import oracle
    cfg = _c2(100)
    G = oracle.layout(cfg)
    hp, (q0, eps0, p0) = chain_state(cfg, 24, np.float32, 5, period)
    ref = oracle.scan(G, q0, eps0, p0, 3, hp=hp, seed=5, trace=True, n_threads=0)
    for p1, p2, n in chain_counts(G, p0, ref.trace_prices):
        if period == 1:
            assert p1 > 0.9 * n, (p1, n)
        else:
            assert p2 >= 300, p2


# ------------------------------------------------------------------------------------------------ GPU
def _device():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    prop = torch.cuda.get_device_properties(0)
    return prop.multi_processor_count, prop.shared_memory_per_block_optin


def _set_kernel(monkeypatch, kernel):
    monkeypatch.delenv("THRL_KERNEL", raising=False)
    monkeypatch.delenv("THRL_LPC_GL", raising=False)
    if kernel == "generic":
        monkeypatch.setenv("THRL_KERNEL", "generic")
    elif kernel.startswith("lpc"):
        monkeypatch.setenv("THRL_KERNEL", "lpc")
        monkeypatch.setenv("THRL_LPC_GL", kernel[3:])


def _check_kernel(cfg, elem, kernel):
    """The kernel that ran is the one the restated plan calls for; on the headline kernel, the resident runs are the
    restated warps per CTA on every SM (thrl_last_wave_runs is set from the plan, before a small batch shrinks the CTA)."""
    from th_rl_b200 import _lib
    sms, optin = _device()
    plan = lut2_plan(cfg, elem, _noisy(cfg), optin)
    got = _lib.last_kernel()
    if kernel == "generic":
        assert got == "generic", got
    elif not planned(plan):
        assert got != "lut2", got
    elif kernel.startswith("lpc") and not _noisy(cfg):
        assert got == "lpc", got
    else:
        assert got == "lut2", got
        assert _lib.last_wave_runs() == sms * plan["warps"], (_lib.last_wave_runs(), sms, plan["warps"])


def _refused(cfg, dtype):
    """The scan raises THRL_ERR_UNSUPPORTED instead of playing the game."""
    import torch
    from th_rl_b200 import engine
    from th_rl_b200._lib import ThrlError
    b = engine.RunBatch(cfg, 4, dtype=torch.float64 if dtype == np.float64 else torch.float32, seed=1).init_device()
    with pytest.raises(ThrlError) as ei:
        b.scan(1)
        torch.cuda.synchronize()
    assert ei.value.code == abi.THRL_ERR_UNSUPPORTED


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["auto", "generic", "lpc8", "lpc16"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_plan_edge_matches_oracle(case, kernel, monkeypatch):
    """Every case, f32 and f64 tables, 40 runs with per-run hyper-parameters, bit for bit against the oracle; on the
    headline kernel where the plan takes the game (the fallback where it does not), on the general kernel, and on the
    lane-per-chain kernel where its layout fits.  A call no kernel can play is refused: the lane-per-chain kernel where its
    layout does not fit, and the general kernel on the episodes of T_MAX steps and more (it keeps per-step state of the
    whole episode in shared memory)."""
    from test_gpu_parity import _philox_case
    cfg, _ = CASES[case]
    if kernel.startswith("lpc") and _noisy(cfg):
        pytest.skip("the lane-per-chain kernel is noise-free: same dispatch as auto")
    _set_kernel(monkeypatch, kernel)
    sms, optin = _device()
    for dtype, elem, seed in ((np.float32, 4, 51), (np.float64, 8, 52)):
        plan = lut2_plan(cfg, elem, _noisy(cfg), optin)
        lpc = kernel.startswith("lpc") and planned(plan)
        if (lpc and not lpc_fits(cfg, elem, int(kernel[3:]), optin)) or (
                case in TOO_LONG_FOR_GENERIC and not lpc and not (kernel == "auto" and planned(plan))):
            _refused(cfg, dtype)
            continue
        _philox_case(cfg, 40, 3, dtype, seed=seed, run_id0=3, hp=True, chunks=[1, 2] if case in CHUNKED else None)
        _check_kernel(cfg, elem, kernel)


def _c2_golden(noise=0.0):
    from conftest import load_golden
    cfg = load_golden("c1_example_2q_seed0")["config"]
    cfg["environment"]["noise_prob"] = noise
    return cfg


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["c2_f32", "c2_f64", "c2n_f32"])
def test_full_ctas_match_oracle(shape, monkeypatch):
    """R = 2 waves + 37 runs: full CTAs, every warp plays two or three runs in turn (the initial slots, the greedy cache,
    the rows word of the initial state and the noise price carried from one run to the next), a ragged last round.  Every
    run and every output against the oracle."""
    from test_gpu_parity import _philox_case
    _set_kernel(monkeypatch, "auto")
    sms, optin = _device()
    cfg = _c2_golden(0.05 if shape.startswith("c2n") else 0.0)
    dtype, elem = (np.float64, 8) if shape.endswith("f64") else (np.float32, 4)
    plan = lut2_plan(cfg, elem, _noisy(cfg), optin)
    wave = sms * plan["warps"]
    _philox_case(cfg, 2 * wave + 37, 3, dtype, seed=61, run_id0=11, hp=True)
    _check_kernel(cfg, elem, "auto")


@pytest.mark.gpu
@pytest.mark.parametrize("noise", [0.0, 0.05])
def test_initial_price_slots_match_oracle(noise, monkeypatch):
    """Initial prices of every kind (see initial_prices) on the gapped grid, f32 and f64, two epochs in one call and in
    two calls; noise-free and on the noisy instantiation (where every row up to the reachable price is staged)."""
    from oracle import oracle
    from test_gpu_parity import _philox_case
    _set_kernel(monkeypatch, "auto")
    cfg = _two(40, GAPS["agents"][0], GAPS["agents"][1], noise=noise)
    game = oracle.layout(cfg)
    p0, _ = initial_prices(GAPS)
    R = len(p0)
    for dtype, elem, seed in ((np.float32, 4, 71), (np.float64, 8, 72)):
        q0, c0, eps0, _ = oracle.init(game, R, seed=seed, dtype=dtype, eps0=abi.eps0_from_config(cfg))
        for chunks in (None, [1, 1]):
            _philox_case(cfg, R, 2, dtype, seed=seed, chunks=chunks, state=(q0, eps0, p0))
            _check_kernel(cfg, elem, "auto")


@pytest.mark.gpu
@pytest.mark.parametrize("grid", ["a21", "a40"])
def test_tied_tables_match_oracle(grid, monkeypatch):
    """Tables full of equal maxima and signed zeros: the first maximum must be chosen alike by the greedy-cache build,
    the refresh of written rows and the > 32-column argmax, and by the oracle."""
    from test_gpu_parity import _philox_case
    _set_kernel(monkeypatch, "auto")
    cfg = _c2(60) if grid == "a21" else _c2(60, actions=(40, 21))
    R = 48
    for dtype, elem, seed in ((np.float32, 4, 81), (np.float64, 8, 82)):
        hp, state = tied_state(cfg, R, dtype, seed)
        _philox_case(cfg, R, 4, dtype, seed=seed, hp=hp, state=state, chunks=[1, 3])
        _check_kernel(cfg, elem, "auto")


@pytest.mark.gpu
@pytest.mark.parametrize("period", [1, 2])
def test_repeated_row_chains_match_oracle(period, monkeypatch):
    """Transitions that bootstrap from the row the previous one (period 1) or the one before it (period 2) just wrote."""
    from test_gpu_parity import _philox_case
    _set_kernel(monkeypatch, "auto")
    cfg = _c2(100)
    for dtype, elem, seed in ((np.float32, 4, 91), (np.float64, 8, 92)):
        hp, state = chain_state(cfg, 40, dtype, seed, period)
        _philox_case(cfg, 40, 3, dtype, seed=seed, hp=hp, state=state)
        _check_kernel(cfg, elem, "auto")


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["rows253", "a255", "T1000", "noisy_T200"])
def test_no_store_outside_buffers_at_plan_edges(case, monkeypatch):
    """test_gpu_parity.test_no_store_outside_buffers on the new shapes: a scan, a sub-range scan and a greedy evaluation
    leave every canary byte around the state and output buffers intact."""
    import torch
    from th_rl_b200 import _lib, engine
    from test_gpu_parity import _GuardedArena
    _set_kernel(monkeypatch, "auto")
    cfg, _ = CASES[case]
    R, E = 37, 2
    b = engine.RunBatch(cfg, R, seed=41).init_device()
    arena = _GuardedArena(torch, 96 << 20, b.device)
    for name in ("q", "counter", "eps", "price", "hp", "mlp", "ring"):
        setattr(b, name, arena.adopt(getattr(b, name)))
    b._zeros = arena.zeros
    b.scan(E, stats=True, trace=True, n_log_runs=3)
    assert _lib.last_kernel() == "lut2", _lib.last_kernel()
    b.scan(1, run_range=(5, 30), stats=True, n_log_runs=2, advance=False)
    b.scan(1, stats=True)
    b.greedy_eval(np.full((R, 2), 3.0))
    torch.cuda.synchronize()
    assert arena.damaged() == 0
