#!/usr/bin/env python
"""Bits and launches of a fixed, seeded sequence of Q-network training calls, for comparing two builds of the library
(QLC_LIB=<path> selects one; each build runs in a process of its own):

    QLC_LIB=old/libqlcuda.so python tools/train_bits.py --dump old.npz --kernels old.json
    python tools/train_bits.py --dump new.npz --kernels new.json
    python tools/train_bits.py --diff old.npz new.npz --diff-kernels old.json new.json

--dump writes, after every call, its losses, TD errors, targets y and the f32 master weights of the trained network.
--kernels runs the sequence again, each call alone under torch.profiler, and writes the names of the kernels (and copies) it
launched. --diff compares two dumps byte for byte; --diff-kernels compares the launches of each call as multisets, with the
names the one-step and the n-step target kernels had before they were merged taken as the merged kernel's name.

The sequence runs on a wrapped ring (37 envs, 16 time slots each, truncating episodes), 3 minibatches of 32 per call, on one
network whose target scratch grows and is reused along the way: qlc_qnet_train with a target network and an index >= len in
every minibatch, qlc_qnet_train_weighted (loss weights and TD errors), qlc_qnet_train_host with targets and with a target
network, and qlc_qnet_train_nstep at n_step 1 and 3, vanilla and double DQN, with y_dev.
"""
import argparse
import collections
import importlib
import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np

BATCH, NB, GAMMA = 32, 3, 0.99


def sequence(run):
    """Calls run(name, fn) for each call of the sequence; fn() makes the call and returns its outputs (dict of arrays)."""
    import torch
    from qnet_train_bench import weights
    q = importlib.import_module("q-learning_b200")
    s = torch.cuda.current_stream().cuda_stream
    dev = torch.device("cuda", 0)
    env = q.BreakoutEnvironment(n_envs=37, seed=3, replay_capacity=37 * 16, max_episode_steps=11)
    env.step_many(np.random.default_rng(3).integers(0, 3, size=(40, 37), dtype=np.uint8))
    n_len = q.ReplayBuffer(env).len()
    rng = np.random.default_rng(7)
    net, target = q.QNetwork(env, weights(11)), q.QNetwork(env, weights(12))
    net.set_adam(lr=1e-3)
    n = BATCH * NB
    idx = rng.integers(0, n_len, size=n).astype(np.uint32)
    beyond = idx.copy()
    beyond[5::BATCH] = n_len + np.arange(NB, dtype=np.uint32) * 40
    wts = rng.uniform(0.1, 1.0, size=n).astype(np.float32)
    y_given = rng.normal(size=n).astype(np.float32)

    def dev_u32(a):
        return torch.as_tensor(a.view(np.int32), device=dev)

    idx_d, beyond_d, wts_d = dev_u32(idx), dev_u32(beyond), torch.as_tensor(wts, device=dev)

    def outputs(with_y=True):
        return [torch.full((k,), float("nan"), device=dev) for k in ((NB, n, n) if with_y else (NB, n))]

    def finish(out):
        torch.cuda.synchronize()
        assert net.error() == 0 and target.error() == 0
        res = {k: v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v) for k, v in out.items()}
        res.update({"w_" + k: v for k, v in net.get_weights().items()})
        return res

    def train_target_net():
        loss = outputs(False)[0]
        net.train_device(beyond_d.data_ptr(), BATCH, NB, None, target, GAMMA, loss.data_ptr(), s)
        return finish({"loss": loss})

    def train_weighted():
        loss, td = outputs(False)
        net.train_weighted_device(idx_d.data_ptr(), wts_d.data_ptr(), BATCH, NB, None, target, GAMMA, loss.data_ptr(), td.data_ptr(), s)
        return finish({"loss": loss, "td": td})

    def host_targets():
        return finish({"loss": net.train(idx, targets=y_given, n_batches=NB)})

    def host_target_net():
        return finish({"loss": net.train(idx, target_net=target, gamma=GAMMA, n_batches=NB)})

    def nstep(n_step, double):
        def call():
            loss, td, y = outputs()
            net.train_nstep_device(beyond_d.data_ptr(), wts_d.data_ptr(), BATCH, NB, target, GAMMA, n_step, double, loss.data_ptr(), td.data_ptr(),
                                   y.data_ptr(), s)
            return finish({"loss": loss, "td": td, "y": y})
        return call

    run("train_target_net_beyond_len", train_target_net)
    run("train_weighted", train_weighted)
    run("train_host_targets", host_targets)
    run("train_host_target_net", host_target_net)
    for n_step in (1, 3):
        for double in (False, True):
            run("train_nstep_n%d_%s" % (n_step, "double" if double else "vanilla"), nstep(n_step, double))
    net.close(); target.close(); env.close()


def dump(path):
    out = {}

    def run(name, fn):
        for k, v in fn().items():
            out[name + "/" + k] = v

    sequence(run)
    np.savez(path, **out)
    print("dumped %d arrays to %s" % (len(out), path))


def kernels(path):
    import torch
    from torch.profiler import DeviceType, ProfilerActivity, profile
    sequence(lambda name, fn: fn())                     # warm-up: module load, scratch growth
    out = {}

    def run(name, fn):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            fn()
        out[name] = sorted(e.name for e in prof.events() if e.device_type == DeviceType.CUDA)

    sequence(run)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print("kernels of %d calls to %s" % (len(out), path))


def diff(a, b):
    A, B = np.load(a), np.load(b)
    assert sorted(A.files) == sorted(B.files), "the dumps hold different arrays"
    bad = [k for k in sorted(A.files) if A[k].tobytes() != B[k].tobytes()]
    print("%d arrays, %d bytes compared; %d differ%s" % (len(A.files), sum(A[k].nbytes for k in A.files), len(bad), (": " + ", ".join(bad)) if bad else ""))
    return not bad


TARGET = re.compile(r"\b(?:td_|nstep_)?target_kernel\b")


def diff_kernels(a, b):
    A, B = (json.load(open(p)) for p in (a, b))
    ok = sorted(A) == sorted(B)
    for name in sorted(A):
        ca, cb = (collections.Counter("target_kernel" if TARGET.search(k) else k for k in x[name]) for x in (A, B))
        same = ca == cb
        ok &= same
        print("%-32s %3d launches %s" % (name, sum(ca.values()), "same" if same else "DIFFER: %s vs %s" % (dict(ca - cb), dict(cb - ca))))
    return ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dump")
    ap.add_argument("--kernels")
    ap.add_argument("--diff", nargs=2)
    ap.add_argument("--diff-kernels", nargs=2)
    args = ap.parse_args()
    ok = True
    if args.dump:
        dump(args.dump)
    if args.kernels:
        kernels(args.kernels)
    if args.diff:
        ok &= diff(*args.diff)
    if args.diff_kernels:
        ok &= diff_kernels(*args.diff_kernels)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
