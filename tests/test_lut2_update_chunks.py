"""The headline kernel's update pass in chunks (qtable_scan_lut2 phase D, DESIGN.md 4.1).  With equal batches the batch is
applied 16 transitions at a time: a full chunk through the unrolled body, the partial last one (L % 16 transitions)
through the loop.  Each case is compared with the oracle bit for bit (per-step traces, tables, counters, epsilon, price,
logs and statistics) with f32 and f64 tables, and must have run on the headline kernel.

Batch lengths around the chunk size take either path alone or both; the chain cases make the last transition of a chunk
write the row that the first transition of the next chunk reads (period 1), or the one after it (period 2)."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_lut2_plan_edges import CHUNK, _two, chain_state, lut2_plan  # noqa: E402

# name -> (episode length T, batch length L of both agents)
CASES = {
    "L15": (100, 15),
    "L16": (100, 16),
    "L17": (100, 17),
    "L31": (100, 31),
    "L32": (100, 32),
    "L33": (100, 33),
    "L48": (100, 48),
    "L100": (100, 100),
    "T128": (128, 128),
}


def _cfg(T, L):
    """the C2 grid (21 x 21 actions, 100 states), a batch of the newest L transitions of the episode per agent"""
    return _two(T, dict(min_memory=L, capacity=L), dict(min_memory=L, capacity=L))


def chunks(L):
    """(full chunks, transitions in the partial last chunk) of a batch of L"""
    return L // CHUNK, L % CHUNK


def test_cases_reach_both_paths():
    """Every case is a noise-free equal-batch game on the headline kernel, with the batch length it is named for; together
    they take the full-chunk path alone, the partial-chunk path alone and both."""
    seen = set()
    for name, (T, L) in CASES.items():
        plan = lut2_plan(_cfg(T, L), 4, False)
        assert "rejected" not in plan and plan["L"] == [L, L], (name, plan)
        full, part = chunks(L)
        seen.add((full > 0, part > 0))
    assert seen == {(True, False), (False, True), (True, True)}
    assert chunks(CASES["T128"][1]) == (8, 0)


def _run(cfg, dtype, seed, **kw):
    import torch
    from th_rl_b200 import _lib
    from test_gpu_parity import _philox_case
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    _philox_case(cfg, 40, 3, dtype, seed=seed, **kw)
    assert _lib.last_kernel() == "lut2", _lib.last_kernel()


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_update_chunks_match_oracle(case, monkeypatch):
    """40 runs with per-run hyper-parameters, three epochs, f32 and f64 tables."""
    monkeypatch.delenv("THRL_KERNEL", raising=False)
    T, L = CASES[case]
    for dtype, seed in ((np.float32, 101 + L), (np.float64, 102 + L)):
        _run(_cfg(T, L), dtype, seed, run_id0=5, hp=True)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [48, 100])
@pytest.mark.parametrize("period", [1, 2])
def test_chains_across_chunk_boundaries_match_oracle(period, L, monkeypatch):
    """Greedy chains whose repeated row crosses every chunk boundary: with period 1 the transition that closes a chunk
    writes the row the next chunk's first transition reads."""
    monkeypatch.delenv("THRL_KERNEL", raising=False)
    cfg = _cfg(L, L)
    for dtype, seed in ((np.float32, 111), (np.float64, 112)):
        hp, state = chain_state(cfg, 40, dtype, seed, period)
        _run(cfg, dtype, seed, hp=hp, state=state)
