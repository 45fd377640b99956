"""How often the two serial chains of the headline kernel (qtable_scan_lut2, DESIGN.md 4.1) could skip their shared-memory
round trip, measured on the oracle's traces of the bench's c2 game (CPU only).

    python scripts/lut2_chain_stats.py [--runs 128] [--windows 3000,6000,8000] [--width 100]

The runs are the first `--runs` runs of bench.py's c2 batch (same init seed, run ids and Philox stream); they are played
from epoch 0 with the oracle (bit-exact with the kernel) and traced over each window of `--width` epochs.  Per window and
agent it prints, over the transitions j of the update batches (compact rows = upd_row of the price, as the kernel computes
them):
  dep1       the row j bootstraps from (row of its next state) is the row j-1 writes
  dep2       ... is the row j-2 writes
  fwd        j-1 or j-2 writes a cell of that row (the share of transitions whose row load has to wait for a store)
  same_cell  j writes the cell j-1 wrote
  states     distinct states (prices) per episode
and, for the rollout, the share of step pairs (t, t+1), t even, in which neither agent explores: the pairs that take the
GJ[s] -> GJ[s'] path.  Exploration draws are independent with P = epsilon of the epoch for each agent and step, so this is
((1 - eps0)(1 - eps1))^2 averaged over the window's epochs (epsilon is the same for every run of the c2 batch).
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import oracle  # noqa: E402
from th_rl_b200 import abi  # noqa: E402


def c2_config():
    # bench.py's c2 game (_qcfg(2, 100, 21, 0.2, 0.4, ...)), restated so that this script does not import the benchmark
    return {"agents": [dict(name="QTable", gamma=0.95, actions=21, states=100, alpha=0.1, eps_end=0.001, epsilon=0.5,
                            eps_step=0.9995, action_range=[0.2, 0.4]) for _ in range(2)],
            "environment": dict(name="NoisyPriceState", noise_prob=0, a=10, b=1, nplayers=2, max_steps=100),
            "training": dict(print_freq=500, epochs=1000)}


def upd_row(price, spec):
    return np.rint(price / spec.max_state * float(spec.states)).astype(np.int64)  # agents.py:47-49 on the f64 state


def window_stats(game, price_in, trace_actions, trace_prices):
    """price_in [R] price before the window's first step; trace_actions [R, E, T, 2]; trace_prices [R, E, T]."""
    R, E, T = trace_prices.shape
    flat = trace_prices.reshape(R, E * T)
    before = np.concatenate([price_in[:, None], flat[:, :-1]], axis=1).reshape(R, E, T)  # state of step t
    out = {}
    for a in range(2):
        s = game.agent[a]
        L = 0 if s.min_memory > s.capacity else min(T, s.capacity)
        j0 = T - L
        cu = upd_row(before, s)[:, :, j0:]   # row transition j writes
        cn = upd_row(trace_prices, s)[:, :, j0:]  # row transition j bootstraps from
        k = trace_actions[:, :, j0:, a]
        d1 = cn[:, :, 1:] == cu[:, :, :-1]
        d2 = cn[:, :, 2:] == cu[:, :, :-2]
        same12 = (cu[:, :, :-2] == cu[:, :, 1:-1]) & (k[:, :, :-2] == k[:, :, 1:-1])  # j-2 and j-1 write one cell
        fwd = d1[:, :, 1:] | (d2 & ~same12)
        out[a] = dict(dep1=d1.mean(), dep2=d2.mean(), fwd=fwd.mean(),
                      same_cell=((cu[:, :, 1:] == cu[:, :, :-1]) & (k[:, :, 1:] == k[:, :, :-1])).mean())
    states = np.mean([len(np.unique(trace_prices[r, e])) for r in range(R) for e in range(E)])
    return out, states


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--runs", type=int, default=128)
    ap.add_argument("--windows", default="3000,6000,8000", help="first epoch of each traced window")
    ap.add_argument("--width", type=int, default=100)
    args = ap.parse_args()
    cfg = c2_config()
    game = oracle.layout(cfg)
    q, c, eps, price = oracle.init(game, args.runs, seed=0, dtype=np.float32, eps0=abi.eps0_from_config(cfg))
    threads = oracle.online_cores()
    epoch = 0
    print("window       eps0    agent  dep1   dep2   fwd    same_cell  states  unforced_pairs")
    for w in sorted(int(x) for x in args.windows.split(",")):
        if w > epoch:  # play up to the window untraced
            res = oracle.scan(game, q, eps, price, w - epoch, epoch_begin=epoch, counter=c, seed=0, n_threads=threads)
            q, c, eps, price, epoch = res.q, res.counter, res.eps, res.price, w
        price_in = price.copy()
        res = oracle.scan(game, q, eps, price, args.width, epoch_begin=epoch, counter=c, seed=0, trace=True, n_threads=threads)
        # epsilon of every epoch of the window (agents.py:78, decayed after each epoch; the same for every run)
        e = eps[0].copy()
        unforced = []
        for _ in range(args.width):
            unforced.append(((1.0 - e[0]) * (1.0 - e[1])) ** 2)
            e = np.array([game.agent[a].eps_end + (e[a] - game.agent[a].eps_end) * game.agent[a].eps_step for a in range(2)])
        st, states = window_stats(game, price_in, res.trace_actions, res.trace_prices)
        for a in range(2):
            print("%5d-%-5d  %.4f  %d      %.3f  %.3f  %.3f  %.3f      %5.1f   %.3f"
                  % (w, w + args.width, eps[0][a], a, st[a]["dep1"], st[a]["dep2"], st[a]["fwd"], st[a]["same_cell"], states,
                     np.mean(unforced)))
        q, c, eps, price, epoch = res.q, res.counter, res.eps, res.price, w + args.width


if __name__ == "__main__":
    main()
