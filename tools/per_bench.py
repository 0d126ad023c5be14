#!/usr/bin/env python
"""Costs of prioritized replay on the device (qlc_per_*), with CUDA events, after warm-up, repeated --reps times (median and
min-max reported):

  * qlc_per_sample (with importance weights) and qlc_per_update for minibatches of 32, 512 and 32,768 on a 1 M-transition
    ring of 4,096 envs (256 time steps, full and wrapped);
  * the lazy sync the first PER call after a step launch pays (an update of 0 items: the sync alone), after a 1-step and a
    64-step launch, at 4,096 and 65,536 envs on a 1 M-transition ring;
  * the closed loop of examples/dqn_breakout_torch.py at --envs with --tensor-core-learner, uniform and --prioritized,
    alternated in the same run.

Prints one JSON line and writes it to --out; the card name and power limit are read in the same run.

    python tools/per_bench.py --out profiles/r04_per.json
"""
import argparse
import importlib
import importlib.util
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np
import torch

from qnet_train_bench import gpu_info, stats

q = importlib.import_module("q-learning_b200")
RING = 1 << 20


def filled_env(n_envs, steps):
    env = q.BreakoutEnvironment(n_envs=n_envs, seed=1, replay_capacity=RING)
    env.step_random_device(steps, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return env


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); fn(); b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--iterations", type=int, default=12)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, power = gpu_info()
    res = {"gpu": name, "power_limit": power, "ring_transitions": RING}
    s = torch.cuda.current_stream().cuda_stream
    dev = torch.device("cuda", 0)

    # sample / update on a full, wrapped 1 M ring of 4,096 envs; the priorities are spread by one update over the whole ring first
    env = filled_env(4096, RING // 4096 + 10)
    per = q.PrioritizedReplay(env)
    n = q.ReplayBuffer(env).len()
    all_idx = torch.arange(n, dtype=torch.int32, device=dev)
    per.update_device(all_idx.data_ptr(), torch.randn(n, device=dev).data_ptr(), n, s)
    for batch in (32, 512, 32768):
        idx = torch.empty(batch, dtype=torch.int32, device=dev)
        w = torch.empty(batch, dtype=torch.float32, device=dev)
        td = torch.randn(batch, device=dev)
        calls = 200 if batch < 32768 else 50
        per.sample_device(batch, 1, 0, 0.5, idx.data_ptr(), w.data_ptr(), s)                  # warm-up
        per.update_device(idx.data_ptr(), td.data_ptr(), batch, s)
        torch.cuda.synchronize()

        def sample():
            for c in range(calls):
                per.sample_device(batch, 1, c, 0.5, idx.data_ptr(), w.data_ptr(), s)

        def update():
            for _ in range(calls):
                per.update_device(idx.data_ptr(), td.data_ptr(), batch, s)

        res["sample_us_batch_%d" % batch] = stats([1e3 * event_ms(sample) for _ in range(args.reps)], calls)
        res["update_us_batch_%d" % batch] = stats([1e3 * event_ms(update) for _ in range(args.reps)], calls)
    res["tree_total_finite"] = bool(np.isfinite(per.read()[1]))
    per.close(); env.close()

    # the lazy sync after a step launch: time from the end of the launch to the end of an update of 0 items
    for n_envs in (4096, 65536):
        env = filled_env(n_envs, RING // n_envs + 10)
        per = q.PrioritizedReplay(env)
        dummy = torch.zeros(1, dtype=torch.int32, device=dev)
        per.update_device(dummy.data_ptr(), dummy.data_ptr(), 0, s)
        for k in (1, 64):
            ms = []
            for _ in range(args.reps * 4):
                env.step_random_device(k, stream=s)
                ms.append(event_ms(lambda: per.update_device(dummy.data_ptr(), dummy.data_ptr(), 0, s)))
            res["sync_us_after_%d_step_launch_%d_envs" % (k, n_envs)] = stats([1e3 * x for x in ms], 1)
        per.close(); env.close()

    # closed loop at --envs: uniform and prioritized alternated
    spec = importlib.util.spec_from_file_location("dqn_breakout_torch", os.path.join(ROOT, "examples", "dqn_breakout_torch.py"))
    ex = importlib.util.module_from_spec(spec); spec.loader.exec_module(ex)
    loops = {False: [], True: []}
    for _ in range(3):
        for prio in (False, True):
            ex.run(args.envs, 2, quiet=True, random_phase_steps=0, tensor_core_learner=True, prioritized=prio)              # warm-up
            out = ex.run(args.envs, args.iterations, quiet=True, random_phase_steps=0, tensor_core_learner=True, prioritized=prio)
            loops[prio].append(1e3 * out["seconds"])
            res["closed_loop_%s_qnet_error" % ("prioritized" if prio else "uniform")] = out["qnet_error"]
            res["closed_loop_%s_env_error_flags" % ("prioritized" if prio else "uniform")] = out["error_flags"]
    res["closed_loop_uniform_ms_per_iteration"] = stats(loops[False], args.iterations)
    res["closed_loop_prioritized_ms_per_iteration"] = stats(loops[True], args.iterations)
    res["closed_loop_prioritized_overhead"] = res["closed_loop_prioritized_ms_per_iteration"]["median"] / res["closed_loop_uniform_ms_per_iteration"]["median"] - 1.0
    res["closed_loop_note"] = ("%d envs, %d iterations, --tensor-core-learner, wall clock of run() after its set-up; one update per iteration on "
                               "envs / 4 minibatches of 32 (prioritized: one stratified minibatch of the same size)" % (args.envs, args.iterations))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
