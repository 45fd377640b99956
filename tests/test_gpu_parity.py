"""CUDA path (through the C ABI) against the golden streams of the reference and against the oracle.

Bars: bit-exact for actions, rewards, prices, counters, epsilon, logs and f64 tables; fp32-storage tables within
1e-6 relative of the reference's f64 tables under teacher forcing, and bit-exact against the oracle's fp32 mode.
"""
import numpy as np
import pytest

from th_rl_b200 import abi

pytestmark = pytest.mark.gpu


@pytest.fixture(params=["auto", "generic", "lpc", "lpc16", "mixed", "pwc"], autouse=True)
def kernel_choice(request, monkeypatch):
    """Every test runs with the default dispatch and with each alternative kernel forced, so all kernels are held to the
    same bar.  Games of the lattice kernel (conftest.uses_lattice_kernel) run three times: default (lattice kernel, float32
    tolerance on the MLP state), "pwc" (interval-table kernel forced, same tolerance) and "mixed" (order-exact kernel,
    bit-exact against the oracle); games of the interval-table kernel (conftest.uses_pwc_kernel) twice: default and "mixed"."""
    from conftest import load_golden, uses_lattice_kernel, uses_pwc_kernel, pwc_can_play
    monkeypatch.delenv("THRL_KERNEL", raising=False)
    monkeypatch.delenv("THRL_LPC_GL", raising=False)
    name = getattr(request.node, "callspec", None) and request.node.callspec.params.get("golden")
    cfg = load_golden(name)["config"] if name else None
    lattice = (cfg is not None and uses_lattice_kernel(cfg)) or request.node.get_closest_marker("lattice_game") is not None
    tolerant = lattice or (cfg is not None and uses_pwc_kernel(cfg))
    if request.param == "mixed" and not tolerant:
        pytest.skip("the order-exact MLP kernel is already the default here")
    if request.param == "pwc" and not (lattice and (cfg is None or pwc_can_play(cfg))):
        pytest.skip("the interval-table kernel is the default here, or does not apply")
    if tolerant and request.param in ("generic", "lpc", "lpc16"):
        pytest.skip("same dispatch as the default for this game")
    if request.param == "generic":
        monkeypatch.setenv("THRL_KERNEL", "generic")
    elif request.param in ("mixed", "pwc"):
        monkeypatch.setenv("THRL_KERNEL", request.param)
    elif request.param.startswith("lpc"):
        monkeypatch.setenv("THRL_KERNEL", "lpc")  # lane-per-chain kernel where it applies (else the general kernel)
        if request.param == "lpc16":
            monkeypatch.setenv("THRL_LPC_GL", "16")
    return request.param


# Lattice kernel vs the order-exact computation (oracle): the same real-number gradient summed in another order (f64
# prefix sums instead of sequential float32).  What is compared:
#  * the gradient itself, through Adam's exp_avg / exp_avg_sq, relative to the moment's max-norm: within 2e-5 for
#    Reinforce (measured <= 9e-7: the float32 summation noise of the ORDER-EXACT side over N = 100..1000 terms) and within
#    3e-4 for ActorCritic (measured <= 8e-5 over 24 runs x 6 updates).  ActorCritic's value head sits at 1000
#    (agents.py:244): one float32 ulp of v(s) is 6e-5, the TD terms d_i = gamma * v(s') - v(s) ~ -20 carry that noise, and
#    the actor weight (N r_j + D) / N^2 with D = sum d_i ~ -N * 20 nearly cancels for the high-reward samples -- the
#    reference's own float32 evaluation has the same sensitivity (any other summation order of v moves it as much);
#  * the weights: within 1e-6 absolute + 1e-6 relative (north_star's "1e-6") -- except that Adam moves a weight by
#    lr * g / (|g| + 1e-8) per step, which turns that noise into a visible difference on the few entries whose gradient is
#    itself of the size of the noise.  Those entries (at most 0.1 % of an agent's weights) may differ by up to a quarter
#    of the distance Adam can have moved them, 0.25 * lr * steps; measured: 1 weight in 1.5e5 at 1e-5 (lr = 2e-4).
PWL_ATOL = 1e-6
PWL_RTOL = 1e-6
PWL_MOMENT_TOL = {1: 2e-5, 2: 3e-4, 3: 3e-4}  # by agent kind: Reinforce, ActorCritic, CAC (value head at 1000 like ActorCritic)


def _lattice(cfg, kernel_choice):
    """The game runs on one of the two re-associating MLP kernels (lattice or interval-table): tolerance instead of bits."""
    from conftest import uses_lattice_kernel, uses_pwc_kernel
    return kernel_choice != "mixed" and (uses_lattice_kernel(cfg) or uses_pwc_kernel(cfg))


# Free-running games with CAC agents: the trajectories themselves differ in the last float32 bits (see _lattice_philox_case)
CAC_TRAJ_ATOL = 2e-5
CAC_TRAJ_RTOL = 2e-5
CAC_TRAJ_MOMENT_SCALE = 4.0  # Adam moments of slightly different sample sets: measured 1.8e-5 of the max-norm, bar 4 x 3e-4


def _mlp_close(game, got, ref, moment_scale=1.0):
    """MLP slabs [R, stride] agree (see the tolerance statement above); step counter and buffer header are equal."""
    from th_rl_b200 import abi as _abi
    for i in range(game.n_agents):
        s = game.agent[i]
        if s.kind == _abi.THRL_AGENT_QTABLE:
            continue
        P, o = _abi.mlp_param_count(s), s.mlp_offset
        hdr = slice(o + 3 * P, o + 3 * P + 3)  # Adam step, buffered transitions, ring head
        assert np.array_equal(got[:, hdr].view(np.uint32), ref[:, hdr].view(np.uint32)), i
        steps = ref[:, o + 3 * P:o + 3 * P + 1].view(np.int32).astype(np.float64)
        for k in (1, 2):  # exp_avg, exp_avg_sq
            m, mr = got[:, o + k * P:o + (k + 1) * P].astype(np.float64), ref[:, o + k * P:o + (k + 1) * P].astype(np.float64)
            scale = np.abs(mr).max(axis=1, keepdims=True) + 1e-30
            assert np.all(np.abs(m - mr) <= moment_scale * PWL_MOMENT_TOL[s.kind] * scale), (i, k, float((np.abs(m - mr) / scale).max()))
        w, wr = got[:, o:o + P].astype(np.float64), ref[:, o:o + P].astype(np.float64)
        err = np.abs(w - wr)
        loose = err > PWL_ATOL + PWL_RTOL * np.abs(wr)
        assert loose.mean() <= 1e-3, (i, float(loose.mean()))
        assert np.all(err <= PWL_ATOL + PWL_RTOL * np.abs(wr) + 0.25 * s.lr * steps), (i, float(err.max()))


def torch_int32():
    import torch
    return torch.int32


def _check_dispatch(cfg):
    """The kernel that just ran is the one the game and THRL_KERNEL call for."""
    import os
    from conftest import uses_lattice_kernel
    from th_rl_b200 import _lib
    forced, got = os.environ.get("THRL_KERNEL"), _lib.last_kernel()
    if any(a["name"] != "QTable" for a in cfg["agents"]):
        from conftest import uses_pwc_kernel
        want = "mixed"
        if forced != "mixed":
            want = "pwl" if uses_lattice_kernel(cfg) and forced != "pwc" else ("pwc" if uses_pwc_kernel(cfg) or forced == "pwc" else "mixed")
        assert got == want, (got, want)
    elif forced == "generic":
        assert got == "generic", got
    else:
        assert got in ("lut2", "lpc", "generic", "hbm"), got


def _mods():
    import torch
    from oracle import oracle
    from th_rl_b200 import engine
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch, oracle, engine


def _cuda_replay(g, rng_mode, dtype, exact=True):
    from test_oracle_golden import golden_inputs
    torch, oracle, engine = _mods()
    cfg = g["config"]
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    b = engine.RunBatch(cfg, 1, dtype=tdt)
    q0, mlp0, u, ra, new_a = golden_inputs(g, b.game, rng_mode, dtype)
    b.load_state(q0, [abi.eps0_from_config(cfg)], [g["p0"]], mlp=mlp0)
    E = g["u"].shape[0]
    out = b.scan(E, rng_mode=rng_mode, replay_u=u[None], replay_ra=ra[None],
                 replay_new_a=None if new_a is None else new_a[None], n_log_runs=1, stats=True, trace=True)
    torch.cuda.synchronize()
    _check_dispatch(cfg)
    if mlp0 is not None:  # the oracle on the same inputs: the MLP slab (weights, Adam state, buffers) must agree bit for bit
        ref = oracle.scan(b.game, q0, [abi.eps0_from_config(cfg)], [g["p0"]], E, rng_mode=rng_mode, replay_u=u[None],
                          replay_ra=ra[None], replay_new_a=None if new_a is None else new_a[None], mlp=mlp0)
        if exact:
            assert np.array_equal(b.mlp.cpu().numpy().view(np.uint32), ref.mlp.view(np.uint32)), "MLP slab differs from the oracle"
        else:
            _mlp_close(b.game, b.mlp.cpu().numpy(), ref.mlp)
    return b, out


def _check_vs_golden(g, b, out, exact_tables=True, mlp_atol=None):
    n = b.game.n_agents
    assert np.array_equal(out.trace_actions[0].cpu().numpy(), g["actions"])
    assert np.array_equal(out.trace_rewards[0].cpu().numpy(), g["rewards"])
    assert np.array_equal(out.trace_prices[0].cpu().numpy(), g["prices"])
    from test_oracle_golden import MLP_ATOL, is_mlp
    tabs, cnts = b.tables(), b.counters()
    sds = b.mlp_state_dicts(0) if b.mlp is not None else None
    for i in range(n):
        if is_mlp(g["config"], i):  # against the reference's torch weights: tolerance (float32, different summation order)
            for k, v in sds[i].items():
                ref = g["mlp_final_%d_%s" % (i, k)]
                err = np.abs(v.numpy().reshape(ref.shape) - ref)
                if mlp_atol is None:
                    assert err.max() < MLP_ATOL, (i, k)
                else:  # lattice kernel against torch: same statement as against the oracle (_mlp_close)
                    loose = err > mlp_atol + PWL_RTOL * np.abs(ref)
                    steps = int(b.mlp[0, b.game.agent[i].mlp_offset + 3 * abi.mlp_param_count(b.game.agent[i])].view(torch_int32()).item())
                    assert loose.mean() <= 1e-3 and err.max() <= mlp_atol + 0.25 * b.game.agent[i].lr * steps, (i, k, float(err.max()))
            continue
        got = tabs[i][0].cpu().numpy().astype(np.float64)
        ref = g["q_final_%d" % i]
        if exact_tables:
            assert np.array_equal(got, ref), "table of agent %d" % i
        else:
            rel = np.max(np.abs(got - ref) / np.abs(ref))
            assert rel < 1e-6, rel  # fp32 storage tolerance stated in BASELINE.json north_star
        assert np.array_equal(cnts[i][0].cpu().numpy().astype(np.float64), g["counter_final_%d" % i])
    qt = [i for i in range(n) if not is_mlp(g["config"], i)]
    assert np.array_equal(b.eps[0].cpu().numpy()[qt], g["eps_trace"][-1][qt])
    assert np.array_equal(out.rewards_log[0].cpu().numpy(), g["rewards_log"])
    assert np.array_equal(out.actions_log[0].cpu().numpy(), g["actions_log"])
    assert b.price[0].item() == g["prices"][-1, -1]


def test_replay_draws_f64_matches_reference(golden, kernel_choice):
    """Recorded exploration draws replayed, greedy actions chosen on the GPU: every output equals the reference."""
    lat = _lattice(golden["config"], kernel_choice)
    b, out = _cuda_replay(golden, abi.THRL_RNG_REPLAY_DRAWS, np.float64, exact=not lat)
    _check_vs_golden(golden, b, out, mlp_atol=PWL_ATOL if lat else None)


def test_replay_actions_f64_matches_reference(golden, kernel_choice):
    lat = _lattice(golden["config"], kernel_choice)
    b, out = _cuda_replay(golden, abi.THRL_RNG_REPLAY_ACTIONS, np.float64, exact=not lat)
    _check_vs_golden(golden, b, out, mlp_atol=PWL_ATOL if lat else None)


def test_replay_actions_f32_within_tolerance(golden, kernel_choice):
    lat = _lattice(golden["config"], kernel_choice)
    b, out = _cuda_replay(golden, abi.THRL_RNG_REPLAY_ACTIONS, np.float32, exact=not lat)
    _check_vs_golden(golden, b, out, exact_tables=False, mlp_atol=PWL_ATOL if lat else None)


def _sweep_hp(rng, R, n):
    hp = np.empty((R, n, 4))
    hp[..., 0] = rng.choice([0.05, 0.1, 0.2, 0.5], size=(R, n))
    hp[..., 1] = rng.choice([0.35, 0.8, 0.95, 0.99], size=(R, n))
    hp[..., 2] = 0.001
    hp[..., 3] = rng.choice([0.9, 0.999, 0.9995], size=(R, n))
    return hp


def _philox_case(cfg, R, E, dtype, seed, run_id0=0, hp=False, chunks=None, state=None):
    """hp: True draws per-run hyper-parameters, an [R, n, 4] array gives them.  state: (q0, eps0, p0) to start from instead
    of the library's initial state."""
    torch, oracle, engine = _mods()
    game = oracle.layout(cfg)
    n = game.n_agents
    rng = np.random.default_rng(seed)
    hpa = hp if isinstance(hp, np.ndarray) else (_sweep_hp(rng, R, n) if hp else None)
    q0, c0, eps0, p0, *rest = oracle.init(game, R, seed=seed, run_id0=run_id0, dtype=dtype, hp=hpa,
                                          eps0=abi.eps0_from_config(cfg))
    if state is not None:
        q0, eps0, p0 = state
    mlp0 = rest[0] if rest else None
    ref = oracle.scan(game, q0, eps0, p0, E, hp=hpa, seed=seed, run_id0=run_id0, stats=True, trace=True, n_threads=0, mlp=mlp0)
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    b = engine.RunBatch(cfg, R, dtype=tdt, seed=seed, run_id0=run_id0, hp=hpa)
    b.load_state(q0, eps0, p0, mlp=mlp0)
    outs = [b.scan(e, n_log_runs=R, stats=True, trace=True) for e in (chunks or [E])]
    torch.cuda.synchronize()
    cat = lambda f, ax: np.concatenate([getattr(o, f).cpu().numpy() for o in outs], axis=ax)
    assert np.array_equal(cat("trace_actions", 1), ref.trace_actions)
    assert np.array_equal(cat("trace_prices", 1), ref.trace_prices)
    assert np.array_equal(cat("trace_rewards", 1), ref.trace_rewards)
    assert np.array_equal(b.q.cpu().numpy(), ref.q)
    assert np.array_equal(b.counter.cpu().numpy().view(np.uint32), ref.counter)
    assert np.array_equal(b.eps.cpu().numpy(), ref.eps)
    assert np.array_equal(b.price.cpu().numpy(), ref.price)
    if mlp0 is not None:
        assert np.array_equal(b.mlp.cpu().numpy().view(np.uint32), ref.mlp.view(np.uint32))
    assert np.array_equal(cat("rewards_log", 1), ref.rewards_log)
    assert np.array_equal(cat("actions_log", 1), ref.actions_log)
    assert np.array_equal(cat("stats", 0), ref.stats)
    return b, ref


def _lattice_philox_case(cfg, R, E, seed, run_id0=0, chunks=None):
    """Free-running lattice kernel vs the oracle.  The sampled actions depend on pi(.|s) through `cumsum > u`, so a 1e-7
    difference in a probability flips an action once in ~1e6 draws and the two runs part ways from there: runs whose whole
    action trace equals the oracle's (required: most of them) must agree in everything else -- rewards, prices and logs bit
    for bit, the MLP state within the stated tolerance.  Splitting the call must not change a single bit."""
    torch, oracle, engine = _mods()
    game = oracle.layout(cfg)
    rng = np.random.default_rng(seed)
    hpa = _sweep_hp(rng, R, game.n_agents) if game.run_stride else None
    q0, c0, eps0, p0, mlp0 = oracle.init(game, R, seed=seed, run_id0=run_id0, dtype=np.float32, hp=hpa, eps0=abi.eps0_from_config(cfg))
    ref = oracle.scan(game, q0, eps0, p0, E, hp=hpa, seed=seed, run_id0=run_id0, stats=True, trace=True, n_threads=0, mlp=mlp0)

    def run(chs, trace=True):
        b = engine.RunBatch(cfg, R, seed=seed, run_id0=run_id0, hp=hpa)
        b.load_state(q0, eps0, p0, mlp=mlp0)
        outs = [b.scan(e, n_log_runs=R, stats=True, trace=trace) for e in chs]
        torch.cuda.synchronize()
        _check_dispatch(cfg)
        cat = lambda f, ax: np.concatenate([getattr(o, f).cpu().numpy() for o in outs], axis=ax)
        res = {f: cat(f, 1) for f in (("trace_actions", "trace_prices", "trace_rewards") if trace else ()) + ("rewards_log", "actions_log")}
        res["stats"] = cat("stats", 0)
        res["mlp"], res["price"] = b.mlp.cpu().numpy(), b.price.cpu().numpy()
        res["q"], res["counter"], res["eps"] = b.q.cpu().numpy(), b.counter.cpu().numpy().view(np.uint32), b.eps.cpu().numpy()
        return res

    o = run([E])
    cac = [i for i in range(game.n_agents) if game.agent[i].kind == abi.THRL_AGENT_CAC]
    disc = [i for i in range(game.n_agents) if i not in cac]
    same = (o["trace_actions"][..., disc] == ref.trace_actions[..., disc]).reshape(R, -1).all(axis=1)
    # a run leaves the oracle's trajectory only when a `cdf > u` comparison falls within float32 rounding of a tie (~1e-7 per
    # draw): over R runs x E epochs x T steps x n agents draws that is at most one run in a few dozen
    assert same.sum() >= R - max(1, R // 24), "too many runs left the oracle's trajectory: %d of %d agree" % (same.sum(), R)
    if cac:
        # A CAC action is a float32 sigmoid(mu + std * z) of head outputs that this kernel sums in another order, so it differs
        # from the oracle's in the last bits, and with it every later price: the trajectories stay within float32 rounding of each
        # other instead of being equal (measured: actions within 3e-6, prices within 5e-6 over 12 epochs).
        fa, fr = o["trace_actions"][..., cac].view(np.float32), ref.trace_actions[..., cac].view(np.float32)
        assert np.abs(fa - fr)[same].max() <= CAC_TRAJ_ATOL, float(np.abs(fa - fr)[same].max())
        for f in ("trace_prices", "trace_rewards", "rewards_log", "actions_log"):
            assert np.allclose(o[f][same], getattr(ref, f)[same], rtol=CAC_TRAJ_RTOL, atol=CAC_TRAJ_ATOL), f
        assert np.allclose(o["price"][same], ref.price[same], rtol=CAC_TRAJ_RTOL, atol=CAC_TRAJ_ATOL)
        assert np.array_equal(o["counter"][same].sum(axis=1), ref.counter[same].sum(axis=1))
        assert np.array_equal(o["eps"][same], ref.eps[same])
        if game.run_stride:  # a QTable agent next to it sees rewards that differ in the last bits
            assert np.allclose(o["q"][same], ref.q[same], rtol=1e-5, atol=1e-5)
        _mlp_close(game, o["mlp"][same], ref.mlp[same], moment_scale=CAC_TRAJ_MOMENT_SCALE)
    else:
        for f in ("trace_prices", "trace_rewards", "rewards_log", "actions_log"):
            assert np.array_equal(o[f][same], getattr(ref, f)[same]), f
        assert np.array_equal(o["price"][same], ref.price[same])
        for f in ("q", "counter", "eps"):  # QTable agents of the same game: bit for bit
            assert np.array_equal(o[f][same], getattr(ref, f)[same]), f
        _mlp_close(game, o["mlp"][same], ref.mlp[same])
        if same.all():
            assert np.array_equal(o["stats"], ref.stats)
    o3 = run([E], trace=False)  # the episode loop without the per-step trace stores is a separate code path
    for f in o3:
        assert np.array_equal(o[f].view(np.uint8), o3[f].view(np.uint8)), "untraced call differs in " + f
    if chunks:
        o2 = run(chunks)
        for f in o:
            assert np.array_equal(o[f].view(np.uint8), o2[f].view(np.uint8)), "chunked call differs in " + f
        o4 = run(chunks, trace=False)
        for f in o4:
            assert np.array_equal(o[f].view(np.uint8), o4[f].view(np.uint8)), "untraced chunked call differs in " + f


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_philox_free_running_matches_oracle(golden, dtype, kernel_choice):
    """Free-running Philox mode, many runs, per-run hyper-parameters: bit-exact against the oracle in both dtypes."""
    E = 6 if golden["config"]["environment"]["nplayers"] > 2 else 10
    mixed = any(a["name"] != "QTable" for a in golden["config"]["agents"])
    if _lattice(golden["config"], kernel_choice):
        if dtype == np.float64:
            pytest.skip("no tables: the table dtype does not enter")
        return _lattice_philox_case(golden["config"], 24, 12, seed=1234, run_id0=7)
    _philox_case(golden["config"], 24 if mixed else 96, 12 if mixed else E, dtype, seed=1234, run_id0=7, hp=True)


def test_chunked_scan_equals_single_call(golden, kernel_choice):
    """Splitting the epoch range over several calls (state and pending transitions carried on the device) changes nothing."""
    mixed = any(a["name"] != "QTable" for a in golden["config"]["agents"])
    if _lattice(golden["config"], kernel_choice):
        return _lattice_philox_case(golden["config"], 12, 11, seed=5, chunks=[1, 3, 7])
    _philox_case(golden["config"], 12 if mixed else 40, 11 if mixed else 9, np.float32, seed=5, chunks=[1, 3, 7] if mixed else [1, 3, 5])


def test_host_buffer_entry_point(golden, kernel_choice):
    """thrl_qtable_scan_host (host buffers, copies inside the call) == oracle."""
    torch, oracle, engine = _mods()
    cfg = golden["config"]
    game = oracle.layout(cfg)
    q0, c0, eps0, p0, *rest = oracle.init(game, 33, seed=9, dtype=np.float32, eps0=abi.eps0_from_config(cfg))
    mlp0 = rest[0] if rest else None
    if _lattice(cfg, kernel_choice):  # held to the oracle by the tests above; here: host entry == device entry, bit for bit
        b = engine.RunBatch(cfg, 33, seed=9)
        b.load_state(q0, eps0, p0, mlp=mlp0)
        dev = b.scan(5, n_log_runs=33, stats=True)
        torch.cuda.synchronize()
        q, cnt, eps, p, mlp = q0.copy(), c0.copy(), eps0.copy(), p0.copy(), mlp0.copy()
        out = engine.scan_host(cfg, q, eps, p, 5, counter=cnt, seed=9, n_log_runs=33, stats=True, mlp=mlp)
        assert np.array_equal(mlp.view(np.uint32), b.mlp.cpu().numpy().view(np.uint32))
        assert np.array_equal(q, b.q.cpu().numpy()) and np.array_equal(cnt, b.counter.cpu().numpy().view(np.uint32))
        assert np.array_equal(eps, b.eps.cpu().numpy()) and np.array_equal(p, b.price.cpu().numpy())
        assert np.array_equal(out.rewards_log, dev.rewards_log.cpu().numpy()) and np.array_equal(out.stats, dev.stats.cpu().numpy())
        return
    ref = oracle.scan(game, q0, eps0, p0, 5, seed=9, stats=True, mlp=mlp0)
    q, eps, p, cnt = q0.copy(), eps0.copy(), p0.copy(), c0.copy()
    mlp = None if mlp0 is None else mlp0.copy()
    out = engine.scan_host(cfg, q, eps, p, 5, counter=cnt, seed=9, n_log_runs=33, stats=True, mlp=mlp)
    assert np.array_equal(q, ref.q) and np.array_equal(cnt, ref.counter)
    if mlp is not None:
        assert np.array_equal(mlp.view(np.uint32), ref.mlp.view(np.uint32))
    assert np.array_equal(eps, ref.eps) and np.array_equal(p, ref.price)
    assert np.array_equal(out.rewards_log, ref.rewards_log) and np.array_equal(out.stats, ref.stats)


def test_host_entry_carries_the_ring(kernel_choice):
    """thrl_qtable_scan_host on a game whose batches span episodes (min_memory > max_steps): the pending transitions travel in
    `ring` between calls, so two calls equal one; without a ring the library refuses instead of silently dropping them."""
    if kernel_choice != "auto":
        pytest.skip("independent of the kernel choice")
    from conftest import load_golden
    from th_rl_b200._lib import ThrlError, check, lib
    import ctypes as C
    torch, oracle, engine = _mods()
    cfg = load_golden("hetero_3q_seed4")["config"]
    game = oracle.layout(cfg)
    assert not game.regular
    q0, c0, eps0, p0 = oracle.init(game, 21, seed=13, dtype=np.float32, eps0=abi.eps0_from_config(cfg))
    ref = oracle.scan(game, q0, eps0, p0, 7, seed=13, stats=True)
    q, eps, p, cnt = q0.copy(), eps0.copy(), p0.copy(), c0.copy()
    o1 = engine.scan_host(cfg, q, eps, p, 3, counter=cnt, seed=13, stats=True)
    o2 = engine.scan_host(cfg, q, eps, p, 4, counter=cnt, seed=13, stats=True, epoch_begin=3, ring=o1.ring)
    assert np.array_equal(q, ref.q) and np.array_equal(cnt, ref.counter) and np.array_equal(eps, ref.eps) and np.array_equal(p, ref.price)
    assert np.array_equal(np.concatenate([o1.stats, o2.stats]), ref.stats)
    a = abi.ThrlScanArgs()  # the raw ABI without a ring: refused
    a.game = C.pointer(game)
    a.n_runs, a.epoch_begin, a.epoch_end, a.table_dtype = 21, 0, 1, abi.THRL_F32
    a.q, a.eps, a.price = q.ctypes.data_as(C.c_void_p), eps.ctypes.data_as(C.c_void_p), p.ctypes.data_as(C.c_void_p)
    with pytest.raises(ThrlError) as ei:
        check(lib().thrl_qtable_scan_host(C.byref(a), 0))
    assert ei.value.code == abi.THRL_ERR_BAD_ARGS


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_device_init_matches_oracle(golden, dtype):
    torch, oracle, engine = _mods()
    cfg = golden["config"]
    game = oracle.layout(cfg)
    q0, c0, eps0, p0, *rest = oracle.init(game, 50, seed=77, run_id0=1000, dtype=dtype, eps0=abi.eps0_from_config(cfg))
    b = engine.RunBatch(cfg, 50, dtype=torch.float64 if dtype == np.float64 else torch.float32, seed=77, run_id0=1000)
    b.init_device()
    torch.cuda.synchronize()
    assert np.array_equal(b.q.cpu().numpy(), q0)
    assert np.array_equal(b.eps.cpu().numpy(), eps0) and np.array_equal(b.price.cpu().numpy(), p0)
    if rest:  # nn.Linear default init for the MLP agents, everything else in their blocks zero
        assert np.array_equal(b.mlp.cpu().numpy().view(np.uint32), rest[0].view(np.uint32))
        sd = next(d for d in b.mlp_state_dicts(3) if d is not None)
        head = next(k for k in sd if k.endswith(".weight") and not k.startswith("fc1"))  # fc_pi / fc_mu: fan_in = 256
        assert sd["fc1.weight"].abs().max() <= 1.0 and sd[head].abs().max() <= 1.0 / 16 and sd[head].std() > 0.02
    # agents.py:29: 12.5/(1-gamma) + N(0,1)
    iq = next((i for i in range(game.n_agents) if game.agent[i].kind == abi.THRL_AGENT_QTABLE), None)
    if iq is not None:
        z = b.tables()[iq].cpu().numpy().astype(np.float64) - 12.5 / (1 - game.agent[iq].gamma)
        assert abs(z.mean()) < 0.05 and abs(z.std() - 1.0) < 0.05


def test_greedy_eval_matches_oracle(golden):
    torch, oracle, engine = _mods()
    cfg = golden["config"]
    game = oracle.layout(cfg)
    q0, c0, eps0, p0, *rest = oracle.init(game, 20, seed=3, dtype=np.float64, eps0=abi.eps0_from_config(cfg))
    mlp0 = rest[0] if rest else None
    rng = np.random.default_rng(0)
    price0 = rng.uniform(0, game.a, size=(20, 3))
    new_a = None
    if game.noise_prob > 0:  # play_game draws demand noise (environments.py:28-31): the intercept of every step is an input
        new_a = np.where(rng.uniform(size=(20, 3, game.max_steps)) < 0.3, rng.uniform(0.7 * game.a, game.a, size=(20, 3, game.max_steps)), game.a)
    ref_a, ref_r = oracle.greedy_eval(game, q0, price0, mlp=mlp0, new_a=new_a)
    b = engine.RunBatch(cfg, 20, dtype=torch.float64)
    b.load_state(q0, eps0, p0, mlp=mlp0)
    a, r = b.greedy_eval(price0, new_a=new_a)
    torch.cuda.synchronize()
    assert np.array_equal(a.cpu().numpy(), ref_a) and np.array_equal(r.cpu().numpy(), ref_r)
    if game.noise_prob > 0:
        # without the stream the Python mirror draws it from numpy's global generator in the environment's order ...
        np.random.seed(5)
        a1, r1 = b.greedy_eval(price0)
        np.random.seed(5)
        drawn = engine.draw_demand_intercepts(game.a, game.noise_prob, 20 * 3 * game.max_steps).reshape(20, 3, game.max_steps)
        ref_a1, ref_r1 = oracle.greedy_eval(game, q0, price0, mlp=mlp0, new_a=drawn)
        torch.cuda.synchronize()
        assert np.array_equal(a1.cpu().numpy(), ref_a1) and np.array_equal(r1.cpu().numpy(), ref_r1)
        # ... and the C entry points without the argument refuse a noisy game instead of playing it noise-free
        import ctypes as C
        from th_rl_b200._lib import lib
        out = torch.zeros((20, 3 * game.max_steps, game.n_agents), dtype=torch.float64, device=b.device)
        p0d = torch.as_tensor(price0).to(b.device)
        rc = lib().thrl_greedy_eval_mlp(C.byref(b.game), 20, b.table_dtype, C.c_void_p(b.q.data_ptr()),
                                        C.c_void_p(b.mlp.data_ptr()) if b.mlp is not None else None, 3, C.c_void_p(p0d.data_ptr()),
                                        C.c_void_p(out.data_ptr()), C.c_void_p(out.data_ptr()), None)
        assert rc == abi.THRL_ERR_UNSUPPORTED


def test_greedy_eval_matches_play_game(golden):
    """thrl_greedy_eval(_mlp) against th_rl/utils.py:27-47 `play_game` recorded from the unmodified reference on the agents
    the golden run saved: scaled actions and rewards of every step, bit for bit (f64 tables, the reference's dtype)."""
    from test_oracle_golden import final_state
    torch, oracle, engine = _mods()
    if "eval_p0" not in golden:
        pytest.skip("no play_game record for this case (CAC, whose get_action raises in the reference)")
    cfg = golden["config"]
    b = engine.RunBatch(cfg, 1, dtype=torch.float64)
    q, mlp = final_state(golden, b.game)
    b.load_state(q, [abi.eps0_from_config(cfg)], [golden["p0"]], mlp=mlp)
    a, r = b.greedy_eval(golden["eval_p0"][None], new_a=golden["eval_new_a"][None] if "eval_new_a" in golden else None)
    torch.cuda.synchronize()
    assert np.array_equal(a[0].cpu().numpy(), golden["eval_actions"])
    assert np.array_equal(r[0].cpu().numpy(), golden["eval_rewards"])


@pytest.mark.lattice_game
def test_c5_bench_shape_matches_oracle(kernel_choice):
    """BASELINE C5 exactly as bench.py runs it (bench._c5_cfg: two ActorCritic agents, constructor min_memory = 1000, i.e.
    N = 1000-transition batches every 10 episodes of T = 100): 21 epochs = two updates per agent.  Lattice kernel within the
    stated float32 tolerance of the oracle, chunked == single call; THRL_KERNEL=mixed bit-equal to the oracle."""
    import bench
    cfg = bench._c5_cfg(21)
    if kernel_choice in ("auto", "pwc"):  # lattice kernel; interval-table kernel forced onto the same game
        _lattice_philox_case(cfg, 24, 21, seed=77, run_id0=3, chunks=[4, 9, 8])
    elif kernel_choice == "mixed":
        _philox_case(cfg, 12, 21, np.float32, seed=77, run_id0=3)
    else:
        pytest.skip("same dispatch as the default for this game")


def test_sharding_is_invisible():
    """Philox counters use global run ids: runs [0,R) in one call == the same runs split over two 'ranks'."""
    torch, oracle, engine = _mods()
    from conftest import load_golden
    cfg = load_golden("c1_example_2q_seed0")["config"]
    R, E = 64, 5
    whole = engine.RunBatch(cfg, R, seed=11).init_device()
    ow = whole.scan(E, stats=True)
    parts = [engine.RunBatch(cfg, R // 2, seed=11, run_id0=k * (R // 2)).init_device() for k in range(2)]
    op = [p.scan(E, stats=True) for p in parts]
    torch.cuda.synchronize()
    assert torch.equal(whole.q, torch.cat([p.q for p in parts]))
    assert torch.equal(whole.counter, torch.cat([p.counter for p in parts]))
    assert torch.equal(ow.stats, op[0].stats + op[1].stats)  # what the NCCL all-reduce computes


def test_full_size_properties():
    """BASELINE C2 at full size (65,536 runs): size-independent invariants + run-to-run determinism."""
    torch, oracle, engine = _mods()
    from conftest import load_golden
    cfg = load_golden("c1_example_2q_seed0")["config"]
    R, E, T = 65536, 4, 100
    outs = []
    for rep in range(2):
        b = engine.RunBatch(cfg, R, seed=2).init_device()
        o = b.scan(E, n_log_runs=R, stats=True)
        torch.cuda.synchronize()
        outs.append((b, o))
    (b, o), (b2, o2) = outs
    assert torch.equal(b.q, b2.q) and torch.equal(b.counter, b2.counter) and torch.equal(o.stats, o2.stats)
    for c in b.counters():  # every transition is counted exactly once (agents.py:76)
        assert torch.all(c.reshape(R, -1).sum(1) == E * T)
    e = 0.5
    for _ in range(E):
        e = 0.001 + (e - 0.001) * 0.9995
    assert torch.all(b.eps == e)
    want = torch.round(o.rewards_log * abi.THRL_STATS_SCALE_SUM).to(torch.int64).sum(0)
    assert torch.equal(o.stats[:, :, 0], want)
    # a sample of the full-size batch against the oracle
    game = oracle.layout(cfg)
    idx = np.arange(0, R, 4099)
    q0, c0, eps0, p0 = oracle.init(game, R, seed=2, dtype=np.float32, eps0=abi.eps0_from_config(cfg))
    for r in idx:
        ref = oracle.scan(game, q0[r:r + 1], eps0[r:r + 1], p0[r:r + 1], E, seed=2, run_id0=int(r))
        assert np.array_equal(b.q[r].cpu().numpy(), ref.q[0])


def _c4_cfg(states, actions, n=8, T=100, lo=0.05, hi=0.15):
    a = dict(name="QTable", gamma=0.95, actions=actions, states=states, alpha=0.1, eps_end=0.001, epsilon=0.5,
             eps_step=0.9995, action_range=[lo, hi])
    return {"agents": [dict(a) for _ in range(n)],
            "environment": dict(name="NoisyPriceState", noise_prob=0, a=10, b=1, nplayers=n, max_steps=T),
            "training": dict(print_freq=500, epochs=3)}


def test_c4_full_shape_matches_oracle(kernel_choice):
    """BASELINE C4 at its real shape (8 agents, 1001x101 tables left in HBM, per-run hyper-parameters): bit-exact vs oracle,
    on the gather / on-chip-walk kernel (default) and on the general kernel."""
    from th_rl_b200 import _lib
    if kernel_choice not in ("auto", "generic"):
        pytest.skip("C4 runs on the HBM kernel or, forced, on the general kernel")
    _philox_case(_c4_cfg(1000, 101), 12, 3, np.float32, seed=21, run_id0=5, hp=True)
    assert _lib.last_kernel() == ("hbm" if kernel_choice == "auto" else "generic")
    _philox_case(_c4_cfg(1000, 101), 6, 2, np.float64, seed=22, hp=True)
    assert _lib.last_kernel() == ("hbm" if kernel_choice == "auto" else "generic")


def _hbm_cfg(agents, T, noise=0.0, a=10):
    base = dict(name="QTable", gamma=0.95, alpha=0.1, eps_end=0.001, epsilon=0.5, eps_step=0.9995, states=400, actions=40,
                action_range=[0.1, 0.3], min_memory=T)
    return {"agents": [dict(base, **x) for x in agents],
            "environment": dict(name="NoisyPriceState", noise_prob=noise, a=a, b=1, nplayers=len(agents), max_steps=T),
            "training": dict(print_freq=500, epochs=3)}


HBM_CASES = {
    # every batch full of repeated cells and rows: greedy from the start (one or two price levels per episode)
    "converged": (_hbm_cfg([dict(epsilon=0.0, eps_end=0.0), dict(epsilon=0.0, eps_end=0.0), dict(epsilon=0.02)], 50), {}),
    # alpha = 1 / gamma = 0.99: the live row max decides every value; rows repeat often (coarse 30-state encode)
    "live_max": (_hbm_cfg([dict(alpha=1.0, gamma=0.99, states=30, actions=128), dict(alpha=0.5, states=2000, actions=9)], 64), {}),
    # capacity < max_steps (only the newest transitions are replayed), an agent that never updates, unequal batches
    "ragged": (_hbm_cfg([dict(capacity=37, min_memory=20), dict(min_memory=500, capacity=100), dict(capacity=80, min_memory=80),
                         dict(states=77, actions=5)], 90), {}),
    # demand noise on (env draws per step), odd episode length, one agent
    "noisy": (_hbm_cfg([dict(states=999, actions=61)], 33, noise=0.3), {}),
    # longest episode the kernel takes; 16 agents
    "long_wide": (_hbm_cfg([dict(states=100, actions=12, action_range=[0.02, 0.05]) for _ in range(16)], 254), {}),
    # the staged gather (bulk copies into a shared-memory ring): ring depths -- a single staging batch, more batches than states
    "ring1": (_hbm_cfg([dict(), dict(actions=33)], 20), {"THRL_HBM_GATHER": "bulk", "THRL_HBM_NB": "1"}),
    "ring8": (_hbm_cfg([dict(), dict(actions=33)], 5), {"THRL_HBM_GATHER": "bulk", "THRL_HBM_NB": "8"}),
    "bulk": (_hbm_cfg([dict(), dict(actions=33), dict(states=50)], 40), {"THRL_HBM_GATHER": "bulk"}),
    "bulk_converged": (_hbm_cfg([dict(epsilon=0.0, eps_end=0.0), dict(epsilon=0.0, eps_end=0.0), dict(epsilon=0.02)], 50), {"THRL_HBM_GATHER": "bulk"}),
    "bulk_ragged": (_hbm_cfg([dict(capacity=37, min_memory=20), dict(min_memory=500, capacity=100), dict(capacity=80, min_memory=80),
                              dict(states=77, actions=5)], 90), {"THRL_HBM_GATHER": "bulk"}),
    "bulk_long_wide": (_hbm_cfg([dict(states=100, actions=12, action_range=[0.02, 0.05]) for _ in range(16)], 254), {"THRL_HBM_GATHER": "bulk"}),
    # ... its comparison path (16-byte vector loads + shared stores instead of bulk copies)
    "ldg": (_hbm_cfg([dict(), dict(actions=33), dict(states=50)], 40), {"THRL_HBM_GATHER": "ldg"}),
    # ... lanes per staged row: a whole row per lane (32 rows per batch) ... a quarter-warp per row (4 rows per batch)
    "lpr1": (_hbm_cfg([dict(), dict(actions=33), dict(states=50, actions=7)], 40), {"THRL_HBM_GATHER": "bulk", "THRL_HBM_LPR": "1"}),
    "lpr4": (_hbm_cfg([dict(), dict(actions=33), dict(states=50, actions=7)], 40), {"THRL_HBM_GATHER": "bulk", "THRL_HBM_LPR": "4"}),
    "lpr8": (_hbm_cfg([dict(actions=128), dict(actions=33), dict(states=50, actions=3)], 40),
             {"THRL_HBM_GATHER": "bulk", "THRL_HBM_LPR": "8", "THRL_HBM_NB": "3"}),
    # register landing (default): no L2 prefetch, deep prefetch; widest and narrowest rows
    "reg_pf0": (_hbm_cfg([dict(actions=128), dict(actions=33), dict(states=50, actions=3)], 40), {"THRL_HBM_PF": "0"}),
    "reg_pf9": (_hbm_cfg([dict(actions=128), dict(actions=33), dict(states=50, actions=3)], 40), {"THRL_HBM_PF": "9"}),
    # dynamic schedule (a run played as several tasks that any warp of its CTA may take): one run per CTA, so consecutive tasks
    # of a run land on different warps and every hand-over goes through the done-counter; then 2-3 runs per CTA, ragged batches,
    # per-run hyper-parameters, one task per epoch
    "dyn_handover": (_hbm_cfg([dict(), dict(actions=33), dict(states=50)], 40), {"THRL_HBM_CHUNK": "3"}),
    "dyn_many": (_hbm_cfg([dict(capacity=37, min_memory=20), dict(min_memory=500, capacity=100), dict(capacity=80, min_memory=80),
                           dict(states=77, actions=5)], 90), {"THRL_HBM_CHUNK": "5", "THRL_HBM_WARPS": "2"}),
    "dyn_noisy": (_hbm_cfg([dict(states=999, actions=61)], 33, noise=0.3), {"THRL_HBM_CHUNK": "2"}),
}


@pytest.mark.parametrize("case", sorted(HBM_CASES))
def test_hbm_kernel_edge_shapes_match_oracle(case, kernel_choice, monkeypatch):
    """Corners of the HBM-resident kernel (thrl_scan_hbm.cuh): batches made of repeated cells / rows, truncated and missing
    batches, demand noise, the longest episode, staging-ring depths, both gather paths, every lanes-per-row split; fp32 and
    f64 tables, chunked calls."""
    from th_rl_b200 import _lib
    if kernel_choice != "auto":
        pytest.skip("the general kernel is held to the same oracle by the other tests")
    cfg, env = HBM_CASES[case]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    R = 6 if case.endswith("long_wide") else (330 if case == "dyn_many" else 20)
    _philox_case(cfg, R, 5, np.float32, seed=61, run_id0=9, hp=(case in ("ragged", "bulk_ragged", "live_max", "dyn_many")),
                 chunks=[2, 3] if case in ("converged", "ragged", "bulk_ragged", "dyn_handover") else None)
    assert _lib.last_kernel() == "hbm", _lib.last_kernel()
    _philox_case(cfg, R, 3, np.float64, seed=62)
    assert _lib.last_kernel() == "hbm", _lib.last_kernel()


def test_wide_action_tables_match_oracle(kernel_choice):
    """More than 128 actions (several columns per lane, the general load loop) and 3 agents; also a 2-agent case with
    200 actions, which exceeds what the specialised kernels take and must fall back to the general one."""
    if kernel_choice not in ("auto", "generic"):
        pytest.skip("wide tables always run on the general kernel")
    _philox_case(_c4_cfg(300, 150, n=3, T=40, lo=0.1, hi=0.3), 20, 4, np.float32, seed=23, hp=True)
    _philox_case(_c4_cfg(120, 200, n=2, T=60, lo=0.2, hi=0.45), 20, 4, np.float32, seed=24)


def _two_agent_cfg(T, a0, a1, env=None):
    base = dict(name="QTable", gamma=0.95, alpha=0.1, eps_end=0.001, epsilon=0.5, eps_step=0.9995, states=100, actions=21,
                action_range=[0.2, 0.4])
    return {"agents": [dict(base, **a0), dict(base, **a1)],
            "environment": dict(dict(name="NoisyPriceState", noise_prob=0, a=10, b=1, nplayers=2, max_steps=T), **(env or {})),
            "training": dict(print_freq=500, epochs=3)}


TWO_AGENT_CASES = {
    "odd_T": _two_agent_cfg(33, dict(min_memory=33, capacity=500), dict(min_memory=20, capacity=500)),
    "short_T": _two_agent_cfg(7, dict(min_memory=5, capacity=50), dict(min_memory=7, capacity=50)),
    "partial_chunks": _two_agent_cfg(100, dict(min_memory=50, capacity=53), dict(min_memory=10, capacity=53)),
    "unequal_batches": _two_agent_cfg(60, dict(min_memory=10, capacity=17), dict(min_memory=40, capacity=45)),
    "one_never_fires": _two_agent_cfg(40, dict(min_memory=30, capacity=40), dict(min_memory=100, capacity=50)),
    "unequal_actions": _two_agent_cfg(50, dict(actions=5, min_memory=50, capacity=500), dict(actions=9, states=37, min_memory=50, capacity=500)),
    "wide_actions": _two_agent_cfg(30, dict(actions=40, states=60, min_memory=30), dict(actions=21, min_memory=30)),
    # demand noise on the specialised kernel: every step a noise step (odd episode length: the rollout is single steps only),
    # most steps (runs of consecutive noise steps, episodes that end on one), and the environment's default 5 %
    "noise_all": _two_agent_cfg(33, dict(min_memory=33, capacity=500), dict(min_memory=20, capacity=500), env=dict(noise_prob=1.0)),
    "noise_most": _two_agent_cfg(100, dict(min_memory=50, capacity=53), dict(min_memory=10, capacity=53), env=dict(noise_prob=0.6)),
    "noise_rare": _two_agent_cfg(100, dict(), dict(actions=9, states=37), env=dict(noise_prob=0.05)),
    "T1": _two_agent_cfg(1, dict(min_memory=1, capacity=1), dict(min_memory=1, capacity=1)),
    "T2": _two_agent_cfg(2, dict(min_memory=2, capacity=2), dict(min_memory=2, capacity=2)),
    "L16": _two_agent_cfg(48, dict(min_memory=16, capacity=16), dict(min_memory=16, capacity=16)),
    "L17": _two_agent_cfg(48, dict(min_memory=17, capacity=17), dict(min_memory=17, capacity=17)),
    "L32": _two_agent_cfg(48, dict(min_memory=32, capacity=32), dict(min_memory=32, capacity=32)),
}


@pytest.mark.parametrize("case", list(TWO_AGENT_CASES))
def test_two_agent_edge_shapes_match_oracle(case, kernel_choice):
    """Shapes that exercise the corners of the specialised 2-agent kernel: odd / tiny episode lengths (rollout tail, a single
    partial update chunk), batches that are not a multiple of the 16-transition chunk, agents whose batches differ in
    length (separate update loops), an agent whose buffer never reaches min_memory, unequal and > 32-column action grids;
    one-step and two-step episodes, batches of exactly one update chunk (its read-ahead reaches the pad), one more, and
    exactly two chunks."""
    from th_rl_b200 import _lib
    cfg = TWO_AGENT_CASES[case]
    for dtype, seed in ((np.float32, 41), (np.float64, 42)):
        _philox_case(cfg, 40, 4, dtype, seed=seed, run_id0=3, hp=(case in ("partial_chunks", "noise_most", "L17")),
                     chunks=[1, 3] if case in ("odd_T", "noise_all", "T1", "L16") else None)
    if kernel_choice == "auto":
        assert _lib.last_kernel() == "lut2", _lib.last_kernel()


def test_host_pipeline_equals_resident_scan(kernel_choice):
    """engine.scan_from_host (bench.py's e2e leg: pinned host state in, chunked launches overlapped with the copies, state
    out) leaves exactly the state and statistics of one resident scan -- with plain chunks and with chunks sized in whole
    multiples of the kernel's resident-run count (thrl_last_wave_runs)."""
    if kernel_choice != "auto":
        pytest.skip("host pipeline is independent of the kernel choice")
    torch, oracle, engine = _mods()
    cfg = _two_agent_cfg(20, dict(min_memory=20), dict(min_memory=20))
    for R, chunks in ((1000, 7), (30000, 3)):
        a = engine.RunBatch(cfg, R, seed=5).init_device()
        b = engine.RunBatch(cfg, R, seed=5).init_device()
        ref = a.scan(2, stats=True)
        host = engine.HostState.from_batch(b)
        if R > 20000:
            b.wave = 148 * 23  # what a full-size launch reports on a B200
        stats, h2d, d2h = engine.scan_from_host(b, host, 2, n_chunks=chunks)
        torch.cuda.synchronize()
        assert h2d == d2h == host.nbytes()
        assert torch.equal(host.q, a.q.cpu()) and torch.equal(host.counter, a.counter.cpu())
        assert torch.equal(host.eps, a.eps.cpu()) and torch.equal(host.price, a.price.cpu())
        assert torch.equal(stats, ref.stats)


def test_initial_price_above_reachable_rows(kernel_choice):
    """The call's initial price may encode to a row the demand curve can never reach again (beyond the greedy-cache bound):
    start every run at p0 close to a, which is far above a - a*sum(lo)."""
    torch, oracle, engine = _mods()
    cfg = _c4_cfg(500, 41, n=4, T=30, lo=0.1, hi=0.2)
    game = oracle.layout(cfg)
    R, E = 16, 3
    q0, c0, eps0, p0 = oracle.init(game, R, seed=31, dtype=np.float32, eps0=abi.eps0_from_config(cfg))
    p0 = np.linspace(9.0, 9.99, R)
    ref = oracle.scan(game, q0, eps0, p0, E, seed=31, trace=True)
    b = engine.RunBatch(cfg, R, seed=31)
    b.load_state(q0, eps0, p0)
    out = b.scan(E, trace=True)
    torch.cuda.synchronize()
    assert np.array_equal(out.trace_actions.cpu().numpy(), ref.trace_actions)
    assert np.array_equal(b.q.cpu().numpy(), ref.q)
    assert np.array_equal(b.counter.cpu().numpy().view(np.uint32), ref.counter)


class _GuardedArena:
    """One device allocation filled with a canary byte; every buffer handed to the library is carved out of it with a
    4 KiB gap on both sides, so a store outside any buffer's bounds shows up as a damaged canary."""

    CANARY, GAP = 0xA5, 4096

    def __init__(self, torch, nbytes, device):
        self.torch = torch
        self.mem = torch.full((nbytes,), self.CANARY, dtype=torch.uint8, device=device)
        self.used = torch.zeros((nbytes,), dtype=torch.bool, device=device)
        self.off = self.GAP

    def zeros(self, shape, dtype, device=None):
        n = int(np.prod(shape)) * self.torch.empty((), dtype=dtype).element_size()
        off = (self.off + 255) // 256 * 256
        assert off + n + self.GAP <= self.mem.numel(), "arena too small"
        self.off = off + n + self.GAP
        self.used[off:off + n] = True
        view = self.mem[off:off + n]
        view.zero_()
        return view.view(dtype).reshape(shape)

    def adopt(self, t):
        if t is None:
            return None
        v = self.zeros(tuple(t.shape), t.dtype)
        v.copy_(t)
        return v

    def damaged(self):
        return int(((self.mem != self.CANARY) & ~self.used).sum().item())


GUARD_CASES = ["c1_example_2q_seed0", "noise_2q_seed3", "hetero_3q_seed4", "overflow_2q_seed5", "c4_8q_seed7",
               "mixed_qr_small_seed9", "mixed_arq_seed12", "mixed_cc_seed14", "mlp_aa_seed15", "mlp_raa_seed17", "noise_qr_seed19",
               "noise_ac_seed20"]


@pytest.mark.parametrize("case", GUARD_CASES)
def test_no_store_outside_buffers(case, kernel_choice):
    """Bounds check without a sanitizer: state and output buffers sit between canary bands; scans (a ragged run count,
    chunked, sub-range) and the greedy evaluation must leave every canary byte intact."""
    from conftest import load_golden
    torch, oracle, engine = _mods()
    cfg = load_golden(case)["config"]
    R, E = 37, 2
    b = engine.RunBatch(cfg, R, seed=41).init_device()
    arena = _GuardedArena(torch, 96 << 20, b.device)
    for name in ("q", "counter", "eps", "price", "hp", "mlp", "ring"):
        setattr(b, name, arena.adopt(getattr(b, name)))
    b._zeros = arena.zeros
    b.scan(E, stats=True, trace=True, n_log_runs=3)
    b.scan(1, run_range=(5, 30), stats=True, n_log_runs=2, advance=False)
    b.scan(1, stats=True)
    b.greedy_eval(np.full((R, 2), 3.0))  # noisy games: the intercepts are drawn by the Python mirror
    torch.cuda.synchronize()
    assert arena.damaged() == 0
