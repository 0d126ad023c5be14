#!/usr/bin/env python
"""Timing of the device-side DQN update (qlc_qnet_train) on the replay ring, with CUDA events, after warm-up, repeated
--reps times (median and spread reported):

  * batch 32 (the reference's shape): us per update for --updates updates in ONE call (n_batches = updates) and as
    separate calls (n_batches = 1 each), beside a torch fp32 train step with the same rules (Huber on Q[a], per-variable
    clipnorm, Keras Adam form) on the same minibatch;
  * batch 32,768: ms per update and TFLOP/s (FLOP counted from the layer shapes below) against the B200's dense bf16 peak;
  * the closed loop of examples/dqn_breakout_torch.py at --envs with --tensor-core-learner against its torch learner.

Prints one JSON line and writes it to --out; the card name and power limit are read in the same run.

    python tools/qnet_train_bench.py --out profiles/r03_qnet_train.json
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

q = importlib.import_module("q-learning_b200")

BF16_PEAK_TFLOPS = 2250.0           # dense bf16, one B200 at 1,000 W (data sheet)
MEASURED_BF16_PEAK_TFLOPS = 1627.0  # dense bf16 tcgen05 rate measured on this card (tools/microbench/mma_rate.cu; the forward's denominator)
# GEMM shapes per observation (M rows per item, N, K) of the forward; the backward repeats each as a weight gradient and,
# except conv1, as a data gradient
LAYERS = [(400, 32, 256), (81, 64, 512), (49, 64, 576), (1, 512, 3136), (1, 3, 512)]


def flop_per_update(batch):
    fwd = sum(2 * m * n * k for m, n, k in LAYERS)
    dgrad = sum(2 * m * n * k for m, n, k in LAYERS[1:])
    return batch * (2 * fwd + dgrad)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        name, power = [s.strip() for s in out.splitlines()[0].split(",")]
        return name, power
    except Exception as e:          # noqa: BLE001 - reported, not hidden
        return "unknown (%s)" % e, "unknown"


def weights(seed):
    rng = np.random.default_rng(seed)
    w = {}
    for name, shape in q.QNET_SHAPES.items():
        if name.endswith("kernel"):
            lim = np.sqrt(6.0 / (int(np.prod(shape[:-1])) + shape[-1]))
            w[name] = rng.uniform(-lim, lim, size=shape).astype(np.float32)
        else:
            w[name] = np.zeros(shape, np.float32)
    return w


def timed(fn, reps):
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return out


def stats(ms_list, per):
    v = np.array(ms_list) / per
    return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max()), "reps": len(v)}


class TorchStep:
    """fp32 torch train step with the library's rules (the comparison column)."""

    def __init__(self, w, dev):
        self.w = {k: torch.from_numpy(v.copy()).to(dev).requires_grad_(True) for k, v in w.items()}
        self.m = {k: torch.zeros_like(v) for k, v in self.w.items()}
        self.v = {k: torch.zeros_like(v) for k, v in self.w.items()}
        self.t = 0

    def __call__(self, x, a, y):
        F = torch.nn.functional
        w = self.w
        for p in w.values():
            p.grad = None
        h = x.permute(0, 3, 1, 2)
        for i in (1, 2, 3):
            h = torch.relu(F.conv2d(h, w["conv%d_kernel" % i].permute(3, 2, 0, 1), w["conv%d_bias" % i], stride={1: 4, 2: 2, 3: 1}[i]))
        h = h.permute(0, 2, 3, 1).reshape(h.shape[0], -1)
        h = torch.relu(h @ w["dense1_kernel"] + w["dense1_bias"])
        qv = h @ w["dense2_kernel"] + w["dense2_bias"]
        F.huber_loss(qv.gather(1, a.unsqueeze(1)).squeeze(1), y, delta=1.0).backward()
        self.t += 1
        alpha = 2.5e-4 * np.sqrt(1 - 0.999 ** self.t) / (1 - 0.9 ** self.t)
        with torch.no_grad():
            for k, p in w.items():
                g = p.grad / torch.clamp(p.grad.norm(), min=1.0)
                self.m[k] += (g - self.m[k]) * 0.1
                self.v[k] += (g * g - self.v[k]) * 0.001
                p -= self.m[k] * alpha / (torch.sqrt(self.v[k]) + 1e-7)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--updates", type=int, default=1024)
    ap.add_argument("--big-batch", type=int, default=32768)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    name, power = gpu_info()
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream().cuda_stream
    env = q.BreakoutEnvironment(n_envs=args.envs, seed=3, replay_capacity=args.envs * 16)
    rng = np.random.default_rng(0)
    env.step_many(rng.integers(0, 3, size=(12, args.envs), dtype=np.uint8))
    rb = q.ReplayBuffer(env)
    w = weights(1)
    net, tgt = q.QNetwork(env, w), q.QNetwork(env, w)
    res = {"gpu": name, "power_limit": power, "envs": args.envs}

    # batch 32: one call of `updates` minibatches vs separate calls; targets from the target network (on the device)
    b, u = 32, args.updates
    idx = torch.from_numpy(rng.choice(rb.len(), size=b * u, replace=True).astype(np.int32)).to(dev)
    one_call = lambda: net.train_device(idx.data_ptr(), b, u, None, tgt, 0.99, None, stream)            # noqa: E731
    def separate():
        for j in range(u):
            net.train_device(idx.data_ptr() + 4 * b * j, b, 1, None, tgt, 0.99, None, stream)
    one_call(); separate(); torch.cuda.synchronize()                                                     # warm-up (allocations, module load)
    res["batch32_one_call_us_per_update"] = stats(timed(one_call, args.reps), u / 1000.0)
    res["batch32_separate_calls_us_per_update"] = stats(timed(separate, args.reps), u / 1000.0)
    smp = rb.get_many(idx[:b].cpu().numpy().astype(np.uint32), q.LAYOUT_F32_BXYH)
    x = torch.from_numpy(smp.state).to(dev)
    a = torch.from_numpy(smp.action.astype(np.int64)).to(dev)
    y = torch.from_numpy(smp.reward).to(dev)
    tstep = TorchStep(w, dev)
    torch.backends.cudnn.benchmark = True
    torch.backends.cudnn.allow_tf32 = False            # an fp32 column: no TF32 in convolutions or matmuls
    torch.backends.cuda.matmul.allow_tf32 = False
    n_torch = 200
    def torch_loop():
        for _ in range(n_torch):
            tstep(x, a, y)
    torch_loop(); torch.cuda.synchronize()
    res["batch32_torch_fp32_us_per_update"] = stats(timed(torch_loop, args.reps), n_torch / 1000.0)
    torch.backends.cudnn.allow_tf32 = True             # back to torch's defaults, which the closed-loop torch learner runs with
    torch.backends.cuda.matmul.allow_tf32 = False

    # batch 32,768: one update per call
    bb = args.big_batch
    big = torch.from_numpy(rng.choice(rb.len(), size=bb, replace=False).astype(np.int32)).to(dev)
    yb = torch.zeros(bb, dtype=torch.float32, device=dev)
    big_step = lambda: net.train_device(big.data_ptr(), bb, 1, yb.data_ptr(), None, 0.99, None, stream)   # noqa: E731
    big_step(); torch.cuda.synchronize()
    st = stats(timed(big_step, args.reps), 1.0)
    fl = flop_per_update(bb)
    res["big_batch"] = bb
    res["big_batch_ms_per_update"] = st
    res["big_batch_flop_per_update"] = fl
    res["big_batch_tflops"] = fl / (st["median"] * 1e-3) / 1e12
    res["big_batch_share_of_datasheet_bf16_peak"] = res["big_batch_tflops"] / BF16_PEAK_TFLOPS
    res["big_batch_share_of_measured_bf16_peak"] = res["big_batch_tflops"] / MEASURED_BF16_PEAK_TFLOPS
    res["qnet_error"] = net.error()
    net.close(); tgt.close(); env.close()

    # closed loop (examples/dqn_breakout_torch.py) at --envs: the tensor-core learner vs the torch learner, the shape bench.py
    # reports as actor_loop_learner (greedy actions every iteration, one update per iteration on envs / 4 minibatches of 32)
    import importlib.util
    spec = importlib.util.spec_from_file_location("dqn_breakout_torch", os.path.join(ROOT, "examples", "dqn_breakout_torch.py"))
    ex = importlib.util.module_from_spec(spec); spec.loader.exec_module(ex)
    iters = 12
    for key, tcl in (("closed_loop_tensor_core_learner", True), ("closed_loop_torch_learner", False)):
        per = []
        for _ in range(3):
            ex.run(args.envs, 2, quiet=True, random_phase_steps=0, tensor_core_learner=tcl)                 # warm-up
            out = ex.run(args.envs, iters, quiet=True, random_phase_steps=0, tensor_core_learner=tcl)
            per.append(1e3 * out["seconds"])
        res[key + "_ms_per_iteration"] = stats(per, iters)
        if tcl:
            res[key + "_qnet_error"] = out["qnet_error"]
            res[key + "_env_error_flags"] = out["error_flags"]
    res["closed_loop_note"] = ("%d envs, %d iterations, wall clock of run() after its set-up (env creation excluded); torch learner with torch defaults "
                               "(cudnn TF32 allowed)" % (args.envs, iters))
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
