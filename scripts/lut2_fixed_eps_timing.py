"""Time the headline kernel (qtable_scan_lut2<float, true>) on the C2 shape with epsilon held fixed, for each epsilon given:
the lane-parallel rollout's cost grows with the exploration steps of an episode (about 200 eps of its 100 steps), so this
shows where it gains and where it falls back to the step-by-step rollout.

    python scripts/lut2_fixed_eps_timing.py [--eps 0.5,0.2,0.1,0.03,0.01,0.001] [--runs 131072] [--epochs 200] [--reps 3]

Each run holds its epsilon for the whole call (eps_end = epsilon).  One JSON line per epsilon: kernel ms per call (CUDA
events, median of --reps after a warm-up call) and agent-steps/s, with the GPU's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--eps", default="0.5,0.2,0.1,0.03,0.01,0.001")
    ap.add_argument("--runs", type=int, default=131072)
    ap.add_argument("--epochs", type=int, default=200)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    import numpy as np
    import torch
    from th_rl_b200 import _lib, engine
    T = 100
    base = dict(name="QTable", gamma=0.95, alpha=0.1, eps_end=0.5, epsilon=0.5, eps_step=0.9995, states=100, actions=21,
                action_range=[0.2, 0.4], min_memory=T, capacity=T)
    cfg = {"agents": [dict(base), dict(base)],
           "environment": dict(name="NoisyPriceState", noise_prob=0, a=10, b=1, nplayers=2, max_steps=T),
           "training": dict(print_freq=500, epochs=a.epochs)}
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    for eps in [float(x) for x in a.eps.split(",")]:
        hp = np.empty((a.runs, 2, 4))
        hp[..., 0], hp[..., 1], hp[..., 2], hp[..., 3] = 0.1, 0.95, eps, 0.9995
        b = engine.RunBatch(cfg, a.runs, dtype=torch.float32, seed=1, hp=hp).init_device()
        b.eps.fill_(eps)
        b.scan(a.epochs)  # warm-up; the tables also leave their initial state
        torch.cuda.synchronize()
        assert _lib.last_kernel() == "lut2", _lib.last_kernel()
        ms = []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            b.scan(a.epochs)
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        med = sorted(ms)[len(ms) // 2]
        print(json.dumps(dict(eps=eps, ms=round(med, 3), ms_all=[round(x, 3) for x in ms],
                              agent_steps_per_s=2 * T * a.runs * a.epochs / (med / 1e3), gpu=gpu[0] if gpu else None)),
              flush=True)


if __name__ == "__main__":
    main()
