#!/usr/bin/env python
"""bench.py — agent-steps/s of the th_rl training hot path on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c4|c5] [--no-extras]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path (thrl_qtable_scan) over the whole batch: RUNS_PER_GPU independent runs x
2 QTable agents x EPOCHS epochs x 100 env steps on every GPU (BASELINE C2 shape; 8 GPUs x 131,072 runs = the
1,048,576 runs of C3).  Runs are independent, so ranks share nothing on the data path (weak scaling); the only
collective is the NCCL all-reduce of the per-epoch cross-run statistics, inside the timed region.

value  = agent-steps of all ranks / max-over-ranks CUDA-event time, state resident in HBM.
e2e    = the same work through the reference-facing C-ABI call with HOST buffers (thrl_qtable_scan_host): tables start in
         page-locked host memory, are copied in, scanned and copied back (tables + counters + epsilon + price + statistics),
         all inside the timed region.
workloads = the same measurement (value, e2e, roofline, clocks) for the other two BASELINE shapes -- c4 (8 agents, tables
         left in HBM) and c5 (MLP agents) -- after the headline workload, in the same JSON line (--no-extras skips them).
--impl reference: the CPU arm = the UNMODIFIED Python reference (oracle/_ref, staged by oracle/stage_reference.py) running
         th_rl.trainer.train_one in one process per host core on a bounded sample of the same workload; when the staged
         reference is missing, the oracle port (oracle/thrl_oracle.c, all host threads).  The port's rate is reported next
         to it either way (`cpu_port`): it is ~10^3 x faster per core than the Python loop and the more conservative baseline.
--dump-outputs DIR: after the timed steps of the headline workload, what its last step left a caller is written to
         DIR/<name>.npy (see dump_outputs), so that two builds run with the same arguments can be compared output for output.

bench.py writes nothing into the tree it runs from (which may be read-only): no bytecode caches either.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MAX_STEPS = 100
DUMP_BYTES = 50_000_000  # --dump-outputs writes about this much at most (plus the .npy headers)


def _qcfg(n, states, actions, lo, hi, epochs, noise_prob=0):
    return {
        "agents": [dict(name="QTable", gamma=0.95, actions=actions, states=states, alpha=0.1, eps_end=0.001, epsilon=0.5,
                        eps_step=0.9995, action_range=[lo, hi]) for _ in range(n)],
        "environment": dict(name="NoisyPriceState", noise_prob=noise_prob, a=10, b=1, nplayers=n, max_steps=MAX_STEPS),
        "training": dict(print_freq=500, epochs=epochs),
    }


def _example_cfg(epochs):
    """th_rl/some_path/configs/example_config.json with `epochs` per step."""
    q = dict(name="QTable", gamma=0.95, actions=21, states=100, alpha=0.1, eps_end=0.001, epsilon=0.5, eps_step=0.9995, action_range=[0.2, 0.4])
    r = dict(name="Reinforce", gamma=0.995, actions=21, states=1, action_range=[0.2, 0.4])
    return {"agents": [q, r], "environment": dict(name="NoisyPriceState", noise_prob=0, a=10, b=1, nplayers=2, max_steps=MAX_STEPS),
            "training": dict(print_freq=500, epochs=epochs)}


def _c4_hp(R, n):
    """BASELINE C4 sweep grid: alpha x eps_step x gamma = 64 points, repeated over the runs (64 seeds each at R = 4096)."""
    import numpy as np
    grid = [(al, g, st) for al in (.05, .1, .2, .5) for st in (.999, .9995, .9999, .99995) for g in (.35, .8, .95, .99)]
    hp = np.empty((R, n, 4))
    for r in range(R):
        al, g, st = grid[r % 64]
        hp[r, :, 0], hp[r, :, 1], hp[r, :, 2], hp[r, :, 3] = al, g, 0.001, st
    return hp


def _c5_cfg(epochs, noise_prob=0):
    a = dict(name="ActorCritic", gamma=0.98, actions=21, states=1, action_range=[0.2, 0.4])  # 1 -> 256 -> {21, 1}, N = 1000
    return {"agents": [dict(a), dict(a)],
            "environment": dict(name="NoisyPriceState", noise_prob=noise_prob, a=10, b=1, nplayers=2, max_steps=MAX_STEPS),
            "training": dict(print_freq=500, epochs=epochs)}


# name -> workload.  `algo_bytes` = algorithmic bytes per agent-step (DESIGN.md 4): Q-table shapes 8*A + 16 (SURVEY 8(d)); c5: the
# update's parameter / Adam read-modify-write (6 x 4 B x 6,166 parameters per 1,000-transition batch) + 32 B of transition ring.
# `e2e_chunks`: launches the host entry point cuts a step into (c4: the step is bound by the 27 GB that cross PCIe each way, so
# six launches that overlap their copies beat two launches of one full round each: 2.15e9 vs 1.73e9 end to end; c5 has only 7
# resident waves per step).
WORKLOADS = {
    "c2": dict(agents=2, runs_per_gpu=131072, epochs=1000, e2e_chunks=12, config=_qcfg(2, 100, 21, 0.2, 0.4, 1000), algo_bytes=184.0,
               bound="smem", hp=None,
               desc="2-agent QTable iterated Cournot/PD game (example_config hyper-parameters, 101x21 tables, max_steps=100), "
                    "%d runs/GPU x %d epochs per step (C2 shape; 8 GPUs = the 1,048,576 runs of C3)",
               kernel="thrl::qtable_scan_lut2<float, true> (persistent, one launch per step)"),
    "c4": dict(agents=8, runs_per_gpu=4096, epochs=500, e2e_chunks=6, config=_qcfg(8, 1000, 101, 0.05, 0.15, 500), algo_bytes=824.0,
               bound="hbm", hp=_c4_hp,
               desc="hyper-parameter sweep (alpha x eps_step x gamma = 64 points x 64 seeds), 8 QTable agents, 1001x101 "
                    "tables left in HBM, max_steps=100, %d runs/GPU x %d epochs per step (C4 shape)",
               kernel="thrl::qtable_scan_hbm<float, false> (persistent, one launch per step; distinct rows of an episode gathered once "
                      "with 16-byte vector loads into registers, L2 prefetch two batches ahead, update chain on chip)"),
    "c5": dict(agents=2, runs_per_gpu=16384, epochs=200, e2e_chunks=8, config=_c5_cfg(200), algo_bytes=180.0, bound="hbm", hp=None,
               desc="2 ActorCritic agents (MLP 1->256->{21,1}, Adam, N=1000 transition batches every 10 episodes), "
                    "%d runs/GPU x %d epochs per step (C5 shape)",
               kernel="thrl::mlp_scan_pwl (persistent, one launch per step; policy LUT per lattice state + sorted-breakpoint "
                      "gradient sweep, f64 accumulation; no dense contraction is left)"),
    # the configuration the reference ships (th_rl/some_path/configs/example_config.json: QTable + Reinforce, noise-free), batched:
    # lattice kernel with the QTable agent's table staged in shared memory (DESIGN.md 4.5, last paragraph)
    "ex": dict(agents=2, runs_per_gpu=32768, epochs=100, e2e_chunks=8, config=_example_cfg(100), algo_bytes=180.0, bound="hbm", hp=None,
               desc="the shipped example_config.json pairing (QTable 101x21 + Reinforce 1->256->21, N=1000), %d runs/GPU x %d epochs per step",
               kernel="thrl::mlp_scan_pwl<float, 2, true, *> (lattice kernel, QTable agent staged in shared memory)"),
    # C2 with the environment's own default demand noise (environments.py:7, noise_prob = 0.05): the noisy instantiation of the
    # headline kernel (DESIGN.md 4.1: every reachable row staged, 13-14 resident runs per SM instead of 23)
    "c2n": dict(agents=2, runs_per_gpu=131072, epochs=500, e2e_chunks=12, config=_qcfg(2, 100, 21, 0.2, 0.4, 500, noise_prob=0.05),
                algo_bytes=184.0, bound="smem", hp=None,
                desc="the C2 game with the environment's default demand noise (noise_prob=0.05), %d runs/GPU x %d epochs per step",
                kernel="thrl::qtable_scan_lut2<float, true, true> (noisy instantiation of the headline kernel)"),
    # the same sweep sized to the persistent grid: 3 full rounds of 12 resident runs x 148 SMs (thrl_last_wave_runs reports the
    # round size so that a caller can do this).  4,096 runs are 2.3 rounds, i.e. three balanced rounds of 9-10 runs per SM.
    "c4w": dict(agents=8, runs_per_gpu=5328, epochs=500, e2e_chunks=0, config=_qcfg(8, 1000, 101, 0.05, 0.15, 500), algo_bytes=824.0,
                bound="hbm", hp=_c4_hp,
                desc="the C4 sweep with the run count a whole multiple of the persistent grid's round (64 points x 83.25 seeds), "
                     "8 QTable agents, 1001x101 tables left in HBM, max_steps=100, %d runs/GPU x %d epochs per step",
                kernel="thrl::qtable_scan_hbm<float, false> (as c4)"),
    # C5 with the environment's own default demand noise (environments.py:7, noise_prob = 0.05): the network input is a continuous
    # price, so the lattice kernel does not apply and the interval-table kernel runs (DESIGN.md 4.7).  algo_bytes: one table row
    # per act (22 head columns x 16 B) + the update's share as for c5.
    "c5n": dict(agents=2, runs_per_gpu=16384, epochs=200, e2e_chunks=8, config=_c5_cfg(200, 0.05), algo_bytes=532.0, bound="hbm", hp=None,
                desc="2 ActorCritic agents (MLP 1->256->{21,1}, Adam, N=1000) with the environment's default demand noise "
                     "(noise_prob=0.05: continuous prices), %d runs/GPU x %d epochs per step (C5 shape, noisy)",
                kernel="thrl::mlp_scan_pwc (persistent, one launch per step; exact per-unit float32 thresholds, per-interval (S1,S0) "
                       "head tables, updates by one sweep over the transitions in interval order; no dense contraction is left)"),
}
EXTRAS = ("c2", "c2n", "c4", "c4w", "c5", "c5n", "ex")
# warp instructions per agent-step from the committed ncu captures (profiles/)
NCU_INSTR = {"c2": 30.4, "c5": 110.5, "c5n": 354.9}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("sm_max_mhz", 1965.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1965.0, 1400.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True).start()
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------ CPU legs
def cpu_port_leg(wl, epochs, n_threads=0, target_seconds=8.0):
    """The oracle port (oracle/thrl_oracle.c) on host cores on a bounded sample of the workload (same config, fewer runs)."""
    import numpy as np
    from oracle import oracle
    from th_rl_b200 import abi
    cfg, n = wl["config"], wl["agents"]
    game = oracle.layout(cfg)
    cores = n_threads if n_threads > 0 else oracle.online_cores()
    eps0 = abi.eps0_from_config(cfg)
    # calibrate on a small sample, then size the timed sample for ~target_seconds
    R0 = (64 if n == 2 else 1) * cores
    q0, c0, e0, p0, *rest = oracle.init(game, R0, seed=0, dtype=np.float32, eps0=eps0)
    t = time.perf_counter()
    oracle.scan(game, q0, e0, p0, 20, n_threads=cores, n_log_runs=0, stats=True, mlp=rest[0] if rest else None)
    rate = R0 * n * 20 * MAX_STEPS / (time.perf_counter() - t)
    R = int(max(cores, min(262144, target_seconds * rate / (n * epochs * MAX_STEPS))))
    q0, c0, e0, p0, *rest = oracle.init(game, R, seed=0, dtype=np.float32, eps0=eps0)
    t = time.perf_counter()
    oracle.scan(game, q0, e0, p0, epochs, n_threads=cores, n_log_runs=0, stats=True, mlp=rest[0] if rest else None)
    dt = time.perf_counter() - t
    return {"value": R * n * epochs * MAX_STEPS / dt, "unit": "agent-steps/s", "cores": cores, "kind": "port",
            "sample": "%d runs x %d epochs x %d steps x %d agents of the workload, fp32-storage oracle port "
                      "(oracle/thrl_oracle.c), %d pthreads, %.1f s" % (R, epochs, MAX_STEPS, n, cores, dt)}, dt


class ReferenceLeg:
    """The unmodified Python reference (oracle/_ref): one train_one per host core per sample, epochs sized for ~target seconds."""

    def __init__(self, wl):
        from oracle import oracle, ref_bench
        self.wl, self.cores = wl, oracle.online_cores()
        self.pool = ref_bench.ReferencePool(self.cores)
        self.epochs = None

    def sample(self, target_seconds):
        cfg, n = self.wl["config"], self.wl["agents"]
        if self.epochs is None:  # calibrate: a handful of epochs
            e0 = 4 if any(a["name"] != "QTable" for a in cfg["agents"]) else 20
            _, dt, _ = self.pool.sample(cfg, e0)
            self.epochs = int(max(e0, min(20000, e0 * target_seconds / max(dt, 1e-3))))
        rate, dt, per_proc = self.pool.sample(cfg, self.epochs)
        return {"value": rate, "unit": "agent-steps/s", "cores": self.cores, "kind": "reference",
                "sample": "th_rl.trainer.train_one (unmodified, oracle/_ref) on the workload's config with epochs=%d: %d processes x "
                          "%d agent-steps, one thread each, slowest process %.1f s" % (self.epochs, self.cores, per_proc, dt)}, dt

    def close(self):
        self.pool.close()


def reference_available():
    from oracle import ref_bench
    return ref_bench.available()


def _state_bytes(cfg, R, layout):
    g = layout(cfg)
    return R * (g.run_stride * 8 + g.mlp_stride * 4)


def config_block(name, wl, runs_per_gpu, epochs, n_gpus, layout):
    return {"workload": wl["desc"] % (runs_per_gpu, epochs), "workload_id": name,
            "runs_per_gpu": runs_per_gpu, "global_runs": runs_per_gpu * n_gpus, "epochs_per_step": epochs,
            "max_steps": MAX_STEPS, "agents": wl["agents"], "table_storage": "fp32 (f64 update arithmetic)",
            "rng": "philox4x32-10", "parallelism": "runs sharded over %d GPU(s), no data-path collective; "
                                                   "NCCL all-reduce of per-epoch statistics" % n_gpus,
            "l2": "per-GPU state (%.1f GB) is far larger than the 126 MB L2" % (_state_bytes(wl["config"], runs_per_gpu, layout) / 1e9)}


def base_line(args, name, wl, n_gpus, layout):
    return {
        "metric": "agent-steps/sec", "unit": "agent-steps/s", "n_gpus": n_gpus, "steps": args.steps,
        "warmup": args.warmup, "higher_is_better": True, "scaling": "strong" if getattr(args, "global_runs", None) else "weak",
        "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": config_block(name, wl, args.runs_per_gpu, args.epochs, n_gpus, layout),
    }


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle
    wl = WORKLOADS[args.workload]
    n_samples = args.warmup + args.steps
    target = max(2.0, min(10.0, 120.0 / n_samples))
    vals, cb = [], None
    leg = ReferenceLeg(wl) if reference_available() else None
    for i in range(n_samples):
        cb, dt = leg.sample(target) if leg else cpu_port_leg(wl, args.epochs, target_seconds=target)
        if i >= args.warmup:
            vals.append((cb["value"], dt))
    if leg:
        leg.close()
    v = statistics.mean(x for x, _ in vals)
    line = base_line(args, args.workload, wl, args.gpus, oracle.layout)
    line.update({"impl": "reference", "value": v, "ms_per_step": 1e3 * statistics.mean(d for _, d in vals),
                 "cpu_baseline": dict(cb, value=v),
                 "e2e": {"value": v, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                 "gpu_launches": 0})
    if leg:
        line["cpu_port"], _ = cpu_port_leg(wl, args.epochs, target_seconds=5.0)
        line["config"]["reference_arm"] = ("the unmodified reference: th_rl/trainer.py:29-110 train_one (oracle/_ref), one process per host "
                                           "core, each step a bounded sample (epochs reduced); cpu_port = the C restatement of the same "
                                           "path on all host threads")
    else:
        line["config"]["reference_arm"] = ("oracle/_ref is not staged: oracle port of th_rl/trainer.py:45-70 + agents.py:59-89 + "
                                           "environments.py:25-39 on host cores; the Python reference itself measured 2.35e4 "
                                           "agent-steps/s/core in the build container (BASELINE.md)")
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------ GPU legs
def _sample(n, k):
    """A fixed (seeded) sorted sample of k of range(n); all of it when k >= n."""
    import numpy as np
    return np.arange(n) if k >= n else np.sort(np.random.default_rng(0).choice(n, k, replace=False))


def dump_outputs(batch, out, dump_dir):
    """Writes what the last scan left its caller, as float32 / float64 .npy files in dump_dir:
    stats.npy        [E, n, 4] f64: per epoch and agent, the sums over the runs of the epoch's mean reward, its square, the mean
                     scaled action and its square (the kernel's fixed-point int64 sums over abi.THRL_STATS_SCALE_*);
    and, for a fixed seeded sample of the runs (this rank's runs when there are several), the state the scan advanced in place:
    q_agent<i>.npy   [S, states+1, actions] table of QTable agent i (the batch's table dtype);
    counter_agent<i>.npy [S, states+1, actions] f64 visit counts of QTable agent i;
    eps.npy [S, n] f64, price.npy [S] f64, mlp.npy [S, mlp_stride] f32 (parameters, Adam state and buffers of the MLP agents).
    A stats array larger than a quarter of DUMP_BYTES keeps a fixed sample of its epochs; the runs fill the rest."""
    import numpy as np
    import torch
    from th_rl_b200 import abi
    os.makedirs(dump_dir, exist_ok=True)
    g, R = batch.game, batch.n_runs
    st = out.stats.cpu().numpy()
    st = st[_sample(st.shape[0], max(1, (DUMP_BYTES // 4) // (st[0].size * 8)))]
    scale = np.array([abi.THRL_STATS_SCALE_SUM, abi.THRL_STATS_SCALE_SQ] * 2)
    np.save(os.path.join(dump_dir, "stats.npy"), st.astype(np.float64) / scale)
    agents = [g.agent[i] for i in range(g.n_agents)]
    cells = sum((s.states + 1) * s.actions for s in agents if s.kind == abi.THRL_AGENT_QTABLE)
    per_run = cells * (batch.q.element_size() + 8) + g.mlp_stride * 4 + (g.n_agents + 1) * 8
    runs = torch.as_tensor(_sample(R, max(1, (DUMP_BYTES - st.nbytes) // per_run)), device=batch.device)
    q, counter = batch.q.index_select(0, runs), batch.counter.index_select(0, runs)
    arrays = {"eps": batch.eps.index_select(0, runs), "price": batch.price.index_select(0, runs)}
    for i, s in enumerate(agents):
        if s.kind == abi.THRL_AGENT_QTABLE:
            arrays["q_agent%d" % i] = abi.table_view(q, s)
            arrays["counter_agent%d" % i] = abi.table_view(counter, s).cpu().numpy().view(np.uint32).astype(np.float64)
    if batch.mlp is not None:
        arrays["mlp"] = batch.mlp.index_select(0, runs)
    for k, a in arrays.items():
        np.save(os.path.join(dump_dir, k + ".npy"), a.cpu().numpy() if torch.is_tensor(a) else a)


def measure(name, wl, R, E, steps, warmup, e2e_chunks, ctx, dump_dir=None):
    """value / e2e / roofline / clocks of one workload on this rank's GPU; collective maxima over ranks.  Returns a dict on
    every rank (rank 0 prints it)."""
    torch, np, dist, engine, _lib = ctx["torch"], ctx["np"], ctx["dist"], ctx["engine"], ctx["_lib"]
    world, rank, dev = ctx["world"], ctx["rank"], ctx["dev"]
    nag = wl["agents"]
    agent_steps_rank = R * nag * E * MAX_STEPS
    hp = wl["hp"](R, nag) if wl["hp"] else None

    batch = engine.RunBatch(wl["config"], R, device=dev, dtype=torch.float32, seed=0, run_id0=rank * R, hp=hp).init_device()
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        out = batch.scan(E, stats=True)
        if world > 1:
            dist.all_reduce(out.stats)  # exact int64 sums: the result does not depend on the sharding
    barrier()
    kernel_name = _lib.last_kernel()
    sampler = ClockSampler(dev.index)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    ev[0].record()
    for i in range(steps):
        kev[i][0].record()  # the scan is launched on torch's current stream, where these events are recorded
        out = batch.scan(E, stats=True)
        kev[i][1].record()
        if world > 1:
            dist.all_reduce(out.stats)
        ev[i + 1].record()
    barrier()
    launches = _lib.launch_count() - launches0
    total_ms = ev[0].elapsed_time(ev[-1])
    kern_ms = statistics.mean(a.elapsed_time(b) for a, b in kev)
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([total_ms, kern_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, kern_ms = t.tolist()
    value = agent_steps_rank * world * steps / (total_ms * 1e-3)
    if dump_dir is not None and rank == 0:
        dump_outputs(batch, out, dump_dir)
    del batch, out
    torch.cuda.empty_cache()

    e2e = (measure_e2e(wl, R, E, min(steps, 3), e2e_chunks, ctx, barrier) if e2e_chunks > 0 else
           {"value": None, "unit": "agent-steps/s", "skipped": "not measured for this entry: see workloads.c4.e2e (c4w) / the 1-GPU line (N > 1)"})
    res = {"value": value, "ms_per_step": total_ms / steps, "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
           "kernel_dispatched": kernel_name}

    hbm_peak, sm_max_mhz, tf_peak, peak_src = measured_peaks()
    per_gpu_rate = agent_steps_rank / (kern_ms * 1e-3)
    achieved = per_gpu_rate * wl["algo_bytes"] / 1e9
    roof = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": None,
            "kernel": wl["kernel"], "kernel_ms": kern_ms, "algorithmic_bytes_per_agent_step": wl["algo_bytes"],
            "algorithmic_bytes_per_launch": agent_steps_rank * wl["algo_bytes"]}
    if name == "c2":
        smem_peak_gbs = 128.0 * 148 * sm_max_mhz * 1e6 / 1e9  # 128 B/clk/SM x 148 SMs x max SM clock (BASELINE.md 3)
        run_stride = sum((a["states"] + 1) * a["actions"] for a in wl["config"]["agents"])
        roof.update({
            "bound": "smem", "peak": smem_peak_gbs, "frac": achieved / smem_peak_gbs,
            "note": "tables are shared-memory resident, so the bound is SM shared-memory bandwidth / issue rate, not HBM "
                    "(BASELINE.md 5: 184 algorithmic B per agent-step; peak = 128 B/clk/SM x 148 SMs x %.0f MHz from "
                    "MEASURED_PEAKS.json, %s). ncu (profiles/): ~31 warp instructions and ~6 shared-memory wavefronts "
                    "per agent-step, LSU data pipe ~52%% busy, issue slots ~70%% busy; HBM sees only the one-off slab "
                    "load/store and the visit counters" % (sm_max_mhz, peak_src),
            "hbm": {"achieved": per_gpu_rate * (2 * run_stride * (4 + 4 + 4) / (nag * 1.0 * E * MAX_STEPS)) / 1e9,
                    "peak": hbm_peak, "unit": "GB/s"},
            # the limiter ncu names: warp-instruction issue.  Instructions per agent-step come from the committed ncu
            # capture of this command (profiles/), the rate is the live one.
            "issue_slots": {"warp_inst_per_agent_step": NCU_INSTR["c2"], "achieved": per_gpu_rate * NCU_INSTR["c2"],
                            "peak": 4 * 148 * sm_max_mhz * 1e6, "unit": "warp-inst/s",
                            "frac": per_gpu_rate * NCU_INSTR["c2"] / (4 * 148 * sm_max_mhz * 1e6)}})
    elif name == "c2n":
        smem_peak_gbs = 128.0 * 148 * sm_max_mhz * 1e6 / 1e9
        roof.update({"bound": "smem", "peak": smem_peak_gbs, "frac": achieved / smem_peak_gbs,
                     "note": "as c2 (184 algorithmic B of shared-memory table traffic per agent-step against 128 B/clk/SM x 148 SMs x %.0f MHz, "
                             "%s); the noisy instantiation stages every row the price can reach, so 13-14 runs are resident per SM instead "
                             "of 23, and ~5 %% of the steps take the f64 noise-step path" % (sm_max_mhz, peak_src)})
    elif name in ("c4", "c4w"):
        roof["note"] = ("tables (3.2 MB per run) stay in HBM; 824 algorithmic B per agent-step = 8*A + 16 (BASELINE.md 5: act row + "
                        "bootstrap row + cell + counter); peak = measured copy bandwidth from MEASURED_PEAKS.json (%s).  The kernel "
                        "moves less than that: the act row is served by an exact greedy-action cache on chip and a row that several "
                        "states of an episode share is fetched once (profiles/: DRAM bytes per agent-step)" % peak_src)
    elif name == "c5n":
        tf = per_gpu_rate * 4.5e4 / 1e12
        roof["note"] = ("per agent-step the kernel must read one interval-table row (22 columns x 16 B) to act, and per update the "
                        "parameters and Adam moments as for c5 (148 B) plus 32 B of transition ring: 532 algorithmic B; peak = measured "
                        "copy bandwidth from MEASURED_PEAKS.json (%s).  HBM is not what limits it: the sequential episode is a chain of "
                        "dependent table-row loads and warp-wide softmaxes, so the limiter is issue slots (issue_slots below, "
                        "instructions per agent-step from the committed ncu capture).  The dense formulation (4.5e4 flop per agent-step "
                        "as per-run GEMMs) is not executed: a 1 -> H -> heads ReLU net of a scalar is piecewise linear, the exact "
                        "gradient comes from prefix sums over the transitions in threshold order (DESIGN.md 4.7); tensor-pipe "
                        "utilisation is 0 by construction" % peak_src)
        roof["dense_formulation"] = {"flop_per_agent_step": 4.5e4, "equivalent_tflops": tf, "bf16_peak_tflops": tf_peak,
                                     "frac": tf / tf_peak}
    else:
        tf = per_gpu_rate * 4.5e4 / 1e12
        roof["note"] = ("bound = HBM: what an update must move is the parameters and both Adam moments, read and written (6 x 4 B x 6,166 "
                        "per 1,000-transition batch = 148 B per agent-step) plus 32 B of transition ring; peak = measured copy bandwidth "
                        "from MEASURED_PEAKS.json (%s).  The dense formulation of this workload (BASELINE.md 5: 4.5e4 flop per agent-step "
                        "as GEMMs) is not executed: the network input is a scalar from a finite price lattice, so pi(.|s) is tabulated "
                        "per state and the exact gradient comes from one sorted-breakpoint sweep (DESIGN.md 4.5); tensor-pipe "
                        "utilisation is 0 by construction" % peak_src)
        roof["dense_formulation"] = {"flop_per_agent_step": 4.5e4, "equivalent_tflops": tf, "bf16_peak_tflops": tf_peak,
                                     "frac": tf / tf_peak}
    if name == "ex":
        roof["note"] = ("as c5: HBM algorithmic bytes of the MLP agent's update (148 B per agent-step of that agent) + transition ring; the "
                        "QTable agent's table lives in shared memory for the call.  Bound by issue slots / latency like c5 (DESIGN.md 4.5)")
    if name in ("c5", "c5n"):
        roof["issue_slots"] = {"warp_inst_per_agent_step": NCU_INSTR[name], "achieved": per_gpu_rate * NCU_INSTR[name],
                               "peak": 4 * 148 * sm_max_mhz * 1e6, "unit": "warp-inst/s",
                               "frac": per_gpu_rate * NCU_INSTR[name] / (4 * 148 * sm_max_mhz * 1e6)}
    try:  # DRAM traffic per launch, measured once with ncu --set full on this exact command (profiles/)
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("c4" if name == "c4w" else name)
        if tr and R == wl["runs_per_gpu"]:  # per agent-step as captured x the agent-steps of this launch
            roof["traffic"] = tr["traffic_bytes_per_agent_step"] * agent_steps_rank
            roof["traffic_source"] = tr["source"]
    except (OSError, ValueError):
        pass
    res["roofline"] = roof
    return res


def measure_f64(wl, R, ctx, E=200, steps=2):
    """Secondary figure: the same workload with float64 tables, the reference's own dtype (bit-exact against it under replay;
    the headline stores float32 and updates in float64).  Half the runs: an f64 run needs twice the shared memory."""
    torch, dist, engine, _lib = ctx["torch"], ctx["dist"], ctx["engine"], ctx["_lib"]
    world, rank, dev = ctx["world"], ctx["rank"], ctx["dev"]
    R = max(1, R // 2)
    batch = engine.RunBatch(wl["config"], R, device=dev, dtype=torch.float64, seed=0, run_id0=rank * R).init_device()
    batch.scan(E, stats=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        out = batch.scan(E, stats=True)
        if world > 1:
            dist.all_reduce(out.stats)
    t1.record()
    torch.cuda.synchronize()
    t = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item()
    kern = _lib.last_kernel()
    del batch, out
    torch.cuda.empty_cache()
    return {"value": R * world * wl["agents"] * E * MAX_STEPS * steps / (ms * 1e-3), "unit": "agent-steps/s", "runs_per_gpu": R,
            "epochs_per_step": E, "steps": steps, "ms_per_step": ms / steps, "kernel_dispatched": kern,
            "note": "float64 tables (the reference's dtype): bit-exact against the reference under replay"}


def measure_e2e(wl, R, E, steps, n_chunks, ctx, barrier):
    """Same metric through the reference-facing boundary: thrl_qtable_scan_host on page-locked host buffers -- tables,
    counters, epsilon, price (and the MLP slab) go host -> device -> scan -> host, statistics come back, all inside the timed
    region; the library cuts the run range into chunks so that the copies overlap the kernel."""
    torch, np, dist, engine = ctx["torch"], ctx["np"], ctx["dist"], ctx["engine"]
    world, rank, dev = ctx["world"], ctx["rank"], ctx["dev"]
    from th_rl_b200 import _lib, abi
    nag = wl["agents"]
    need = _state_bytes(wl["config"], R, _lib.game_layout) + R * (nag + 1) * 8  # pinned host copy of tables + counters + eps + price
    try:
        avail = int(next(l for l in open("/proc/meminfo") if l.startswith("MemAvailable")).split()[1]) * 1024
    except (OSError, StopIteration):
        avail = 1 << 62
    if need * world * 2 > avail:
        return {"value": None, "unit": "agent-steps/s", "h2d_bytes_per_step": need * world, "d2h_bytes_per_step": need * world,
                "skipped": "host has %.0f GB available, the pinned state needs %.0f GB" % (avail / 1e9, need * world / 1e9)}
    hp = wl["hp"](R, nag) if wl["hp"] else None
    batch = engine.RunBatch(wl["config"], R, device=dev, dtype=torch.float32, seed=1, run_id0=rank * R, hp=hp).init_device()
    torch.cuda.synchronize()
    host = engine.HostState.from_batch(batch)  # pinned host copies of q / counter / eps / price (/ mlp)
    del batch
    torch.cuda.empty_cache()
    q, eps, price = host.q.numpy(), host.eps.numpy(), host.price.numpy()
    counter = host.counter.numpy().view(np.uint32)
    mlp = None if host.mlp is None else host.mlp.numpy()
    os.environ["THRL_HOST_CHUNKS"] = str(n_chunks)
    epoch = 0
    for it in range(1 + steps):  # one warm-up
        if it == 1:
            barrier()
            t0 = time.perf_counter()
        out = engine.scan_host(wl["config"], q, eps, price, E, counter=counter, hp=hp, seed=1, run_id0=rank * R,
                               epoch_begin=epoch, stats=True, device=dev.index, mlp=mlp)
        epoch += E
        stats = out.stats  # the step's result (per-epoch cross-run statistics) is on the host when the call returns
        if world > 1:
            s = torch.from_numpy(stats).to(dev)
            dist.all_reduce(s)
            stats = s.cpu().numpy()
    barrier()
    dt = time.perf_counter() - t0
    os.environ.pop("THRL_HOST_CHUNKS", None)
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = t.item()
    nb = host.nbytes() + (0 if hp is None else hp.nbytes)
    _lib.lib().thrl_release_device_memory()
    return {"value": R * world * nag * E * MAX_STEPS * steps / dt, "unit": "agent-steps/s",
            "h2d_bytes_per_step": int(nb) * world, "d2h_bytes_per_step": int(host.nbytes() + stats.nbytes) * world,
            "steps": steps, "ms_per_step": 1e3 * dt / steps, "chunks": n_chunks,
            "api": "thrl_qtable_scan_host (C ABI, include/thrl.h) via th_rl_b200.engine.scan_host: page-locked host state in, "
                   "tables+counters+eps+price+stats out"}


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from th_rl_b200 import _lib, engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = dict(torch=torch, np=np, dist=dist, engine=engine, _lib=_lib, world=world, rank=rank, dev=dev)
    wl = WORKLOADS[args.workload]
    res = measure(args.workload, wl, args.runs_per_gpu, args.epochs, args.steps, args.warmup, args.e2e_chunks, ctx,
                  dump_dir=args.dump_outputs)
    line = base_line(args, args.workload, wl, world, _lib.game_layout)
    line.update(res)
    line["parity"] = "green: tests/ -m gpu compare this path with the oracle and the reference's recorded goldens (bit-exact)"
    if args.workload == "c2" and not args.no_extras:
        line["f64_tables"] = measure_f64(wl, args.runs_per_gpu, ctx)
    if not args.no_extras:
        line["workloads"] = {}
        for name in EXTRAS:
            if name == args.workload:
                continue
            w2 = WORKLOADS[name]
            # the host round trip of the secondary workloads is measured on one GPU only: at N ranks their pinned host copies
            # (c4: 27 GB per rank) would have to coexist in one box's memory for a number that the N = 1 line already carries
            try:
                r2 = measure(name, w2, w2["runs_per_gpu"], w2["epochs"], min(args.steps, 3), 3, w2["e2e_chunks"] if world == 1 else 0, ctx)
            except Exception as exc:  # a secondary workload must not cost the headline line (one process: no collective to desynchronise)
                if world > 1:
                    raise
                torch.cuda.empty_cache()
                line["workloads"][name] = {"error": "%s: %s" % (type(exc).__name__, str(exc)[:300])}
                continue
            r2["config"] = config_block(name, w2, w2["runs_per_gpu"], w2["epochs"], world, _lib.game_layout)
            r2["steps"], r2["warmup"], r2["unit"] = min(args.steps, 3), 3, "agent-steps/s"
            line["workloads"][name] = r2
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        if args.no_cpu_baseline:
            line["cpu_baseline"] = None
        else:
            line["cpu_port"], _ = cpu_port_leg(wl, args.epochs, target_seconds=8.0)
            if reference_available():
                leg = ReferenceLeg(wl)
                line["cpu_baseline"], _ = leg.sample(10.0)
                leg.close()
            else:
                line["cpu_baseline"] = line["cpu_port"]
        print(json.dumps(line))


def main():
    # no bytecode caches in the tree, from this process or the ones it starts (torchrun ranks, reference workers)
    sys.dont_write_bytecode = True
    os.environ["PYTHONDONTWRITEBYTECODE"] = "1"
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS),
                    help="c2 = headline (default); c4 = HBM-resident sweep; c5 = MLP (ActorCritic) agents; c5n = c5 with demand noise")
    ap.add_argument("--global-runs", type=int, default=None,
                    help="total runs of the job, split evenly over the ranks (strong scaling; BASELINE config 3 = 1048576)")
    ap.add_argument("--runs-per-gpu", type=int, default=None)
    ap.add_argument("--epochs", type=int, default=None)
    ap.add_argument("--e2e-chunks", type=int, default=None, help="launches the host entry point cuts a step into (default: per workload)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the c4 / c5 measurements that follow the headline workload")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the headline workload's last timed step computed to DIR/<name>.npy (at most ~50 MB: a fixed sample of the runs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    wl = WORKLOADS[args.workload]
    if args.global_runs:
        args.runs_per_gpu = args.global_runs // max(1, args.gpus)
    args.runs_per_gpu = args.runs_per_gpu or wl["runs_per_gpu"]
    args.epochs = args.epochs or wl["epochs"]
    args.e2e_chunks = wl["e2e_chunks"] if args.e2e_chunks is None else args.e2e_chunks
    if args.impl == "reference":
        return run_reference(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: relaunch under torchrun
        port = 29500 + os.getpid() % 1000
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(port)] + sys.argv
        sys.exit(subprocess.call(cmd))
    run_ours(args)


if __name__ == "__main__":
    main()
