#!/usr/bin/env python
"""Costs of n-step returns and double-DQN targets on the device (DESIGN.md §14), with CUDA events, after warm-up, repeated
--reps times (median and min-max reported):

  * qlc_replay_nstep for 32 and 32,768 items with n_step 1, 3 and 10, on a wrapped 1 M-transition ring of 4,096 envs;
  * qlc_qnet_train_nstep (vanilla n = 3, double DQN n = 3) against qlc_qnet_train, one update of a minibatch of 32 and of
    32,768 per call, the three alternated in the same run.

Prints one JSON line and writes it to --out; the card name and power limit are read in the same run.

    python tools/nstep_bench.py --out profiles/r05_nstep.json
"""
import argparse
import importlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np
import torch

from qnet_train_bench import gpu_info, stats, timed, weights

q = importlib.import_module("q-learning_b200")
RING, N_ENVS = 1 << 20, 4096


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, power = gpu_info()
    res = {"gpu": name, "power_limit": power, "ring_transitions": RING, "n_envs": N_ENVS}
    s = torch.cuda.current_stream().cuda_stream
    dev = torch.device("cuda", 0)
    env = q.BreakoutEnvironment(n_envs=N_ENVS, seed=1, replay_capacity=RING, max_episode_steps=10_000)
    env.step_random_device(RING // N_ENVS + 10, stream=s)                    # full and wrapped
    rb = q.ReplayBuffer(env)
    n_len = rb.len()
    gen = torch.Generator(device=dev); gen.manual_seed(0)

    # qlc_replay_nstep
    for n in (32, 32768):
        idx = torch.randint(0, n_len, (n,), dtype=torch.int32, device=dev, generator=gen)
        G, d, b = (torch.empty(n, dtype=torch.float32, device=dev), torch.empty(n, dtype=torch.float32, device=dev), torch.empty(n, dtype=torch.int32, device=dev))
        for n_step in (1, 3, 10):
            calls = 500

            def run():
                for _ in range(calls):
                    rb.nstep_device(idx.data_ptr(), n, n_step, 0.99, G.data_ptr(), d.data_ptr(), b.data_ptr(), s)

            run()
            res["replay_nstep_us_items_%d_n_%d" % (n, n_step)] = stats([1e3 * x for x in timed(run, args.reps)], calls)

    # qlc_qnet_train vs qlc_qnet_train_nstep, vanilla and double, alternated
    online, target = q.QNetwork(env, weights(1)), q.QNetwork(env, weights(2))
    for batch in (32, 32768):
        calls = 40 if batch == 32 else 4
        idx = torch.randint(0, n_len, (calls, batch), dtype=torch.int32, device=dev, generator=gen)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        kinds = {
            "train": lambda i: online.train_device(idx[i].data_ptr(), batch, 1, None, target, 0.99, loss.data_ptr(), s),
            "nstep3": lambda i: online.train_nstep_device(idx[i].data_ptr(), None, batch, 1, target, 0.99, 3, False, loss.data_ptr(), None, None, s),
            "nstep3_double": lambda i: online.train_nstep_device(idx[i].data_ptr(), None, batch, 1, target, 0.99, 3, True, loss.data_ptr(), None, None, s),
        }
        ms = {k: [] for k in kinds}
        for _ in range(args.reps + 1):
            for k, f in kinds.items():
                ms[k].append(timed(lambda: [f(i) for i in range(calls)], 1)[0])
        for k in kinds:
            res["%s_us_per_update_batch_%d" % (k, batch)] = stats([1e3 * x for x in ms[k][1:]], calls)     # the first round warms up
        base = res["train_us_per_update_batch_%d" % batch]["median"]
        for k in ("nstep3", "nstep3_double"):
            res["%s_over_train_batch_%d" % (k, batch)] = res["%s_us_per_update_batch_%d" % (k, batch)]["median"] / base - 1.0
    res["qnet_error"] = online.error() | target.error()
    res["env_error_flags"] = env.error_flags()
    online.close(); target.close(); env.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
