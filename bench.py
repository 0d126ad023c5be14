#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (BASELINE.json): Breakout env-steps/s
(step + render + 84x84 u8 preprocess + 4-frame stack append + replay insert) and replay-sampled transitions/s.

    python bench.py --gpus 1 --steps K --warmup W                  # this repo's CUDA path
    python bench.py --impl reference --gpus 1 --steps K --warmup W # the restated reference CPU path (oracle)
    torchrun ... bench.py --gpus N ...                             # one rank per GPU, env shards, no data-path collective
    python bench.py ... --dump-outputs DIR                         # also write what the last timed step computed, DIR/<name>.npy

One bench "step" = ONE launch of the fused kernel advancing every env of the shard by STEPS_PER_LAUNCH env-steps
on a synthetic action stream (config.workload says which). Prints ONE JSON line (rank 0).
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

ENVS_PER_GPU = 4096            # BASELINE.json configs[1]
STEPS_PER_LAUNCH = 64          # env-steps per env per launch: 4096*64*7056 B = 1.85 GB of frames per bench step (>> 126 MB L2)
REPLAY_CAPACITY = 1 << 20      # 1M transitions (configs[2]) = 256 time steps of 4096 envs, 7.4 GB of frames
BYTES_PER_ENV_STEP = 7066      # frame 7,056 + action 1 + reward 4 + done 1 + replay record 4 (SURVEY.md 8(d) minus the per-launch state)
STATE_BYTES_PER_ENV = 53       # 7 f32 + u64 brick mask + 4 u32 + 1 u8: read once and written once per LAUNCH, not per step
BYTES_PER_SAMPLE_U8 = 91744    # 5 frames read + 2 x 4 frames written + 16 B scalars
BYTES_PER_SAMPLE_F32 = 261088  # 5 frames read + 2 x 4 f32 frames written + 16 B scalars
SEED = 20261018
SETTLE_LAUNCHES = 1000         # untimed launches after the warm-up: 0.29 s of the default config (0.286 ms per launch, B200 at a 1,000 W power limit)
DUMP_OBS_ENVS = 256            # --dump-outputs: envs whose observation stacks are written, 256 x 112,896 B of f32
QNET_FLOP_PER_OBS = 2 * (400 * 32 * 256 + 81 * 64 * 512 + 49 * 64 * 576 + 512 * 3136 + 3 * 512)   # 84x84x4 -> conv 8/4, 4/2, 3/1 -> 512 -> 3


def launch_bytes(n_envs, k_inner):
    """algorithmic bytes of ONE step launch, exact: 7,066 B per env-step + 2 x 53 B of env state per env"""
    return BYTES_PER_ENV_STEP * n_envs * k_inner + 2 * STATE_BYTES_PER_ENV * n_envs


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _ncu_traffic(kernel):
    """dram bytes per launch from the committed ncu --set full capture, if one exists."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(kernel)
        except Exception:
            return None
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the GPU is under load (B200_PROFILING.md recipe)."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in self.rows:
            c = [x.strip() for x in r.split(",")]
            if len(c) < 8:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(names, c[4:8]):
                if v == "Active":
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _config(n_envs, k_inner, replay_capacity, world):
    """the workload both arms name: BASELINE.json configs[1] (4,096 envs on one B200) with the configs[2] replay ring behind it"""
    return {"workload": "%d Breakout envs per GPU: step+render+84x84 u8 frame+4-frame stack append+replay insert, %d env-steps per launch, uniform random action stream" % (n_envs, k_inner),
            "envs_per_gpu": n_envs, "steps_per_launch": k_inner, "replay_capacity": replay_capacity,
            "l2": "each step writes %.2f GB of frames (> 126 MB L2); ring of %.1f GB" % (n_envs * k_inner * 7056 / 1e9, (replay_capacity // n_envs + 4) * n_envs * 7056 / 1e9),
            "parallelism": "env-sharded x%d, no data-path collective" % world}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path. The Rust crate cannot be built in this image
    (no cargo/rustc; its renderer is unimplemented!()), so this times the oracle port on all host cores."""
    if rank != 0:
        return
    from oracle import oracle as O
    O.build()
    cores = os.cpu_count() or 1
    # one step = one whole bench step on the CPU (every env, every env-step) whenever K of them fit in about two minutes on this
    # box's cores; a longer run takes a bounded sample of each step: every env, fewer of its env-steps
    sample_envs = args.envs
    O.bench_env_steps(sample_envs, 2, SEED, cores)                              # spin the thread pool up once, outside the timed steps
    probe = O.bench_env_steps(sample_envs, 4, SEED, cores)
    rate = sample_envs * 4 / max(probe, 1e-9)
    sample_steps = int(max(1, min(args.steps_per_launch, 120.0 * rate / (max(args.steps, 1) * sample_envs))))
    for _ in range(args.warmup):
        O.bench_env_steps(sample_envs, max(1, sample_steps // 8), SEED, cores)
    t = 0.0
    for _ in range(args.steps):
        t += O.bench_env_steps(sample_envs, sample_steps, SEED, cores)
    units = sample_envs * sample_steps * args.steps
    value = units / t
    sample = ("each step = %d envs x %d env-steps (%s bench step of the same workload: step+render+grayscale+4-frame ring+per-step state clone, "
              "the reference's CPU path restated in C), %d OpenMP threads" % (sample_envs, sample_steps,
                                                                               "ONE whole" if sample_steps == args.steps_per_launch else "%d/%d of a" % (sample_steps, args.steps_per_launch), cores))
    line = {
        "impl": "reference", "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config(args.envs, args.steps_per_launch, args.replay_capacity, max(1, args.gpus)),      # the B200 arm's config at this N, verbatim
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_b200(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    q = importlib.import_module("q-learning_b200")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    distributed = world > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG / NCCL_DEBUG_FILE are left as the launcher set them (the driver reads the rank count out of NCCL's log);
        # the JSON line is the LAST line rank 0 writes to stdout.
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    build = q.build_info()
    if build.get("profiling") != "0":
        raise SystemExit("bench.py: libqlcuda.so is an ablation build (-DQLC_PROFILING honours QLC_DEBUG_SKIP); bench numbers need the release build")
    n_envs, k_inner = args.envs, args.steps_per_launch
    env = q.BreakoutEnvironment(n_envs=n_envs, seed=SEED, env_id_base=rank * n_envs,   # = sharding.shard_range(rank, world, world * n_envs)[0]
                                replay_capacity=args.replay_capacity, device=local_rank)
    rb = q.ReplayBuffer(env)
    gen = torch.Generator(device=dev); gen.manual_seed(SEED + rank)
    actions = torch.randint(0, 3, (k_inner, n_envs), dtype=torch.uint8, device=dev, generator=gen)   # synthetic action stream, resident in HBM
    reward = torch.empty((k_inner, n_envs), dtype=torch.float32, device=dev)
    done = torch.empty((k_inner, n_envs), dtype=torch.uint8, device=dev)
    stats_vec = torch.zeros(5, dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def launch():
        env.step_device(actions.data_ptr(), k_inner, reward.data_ptr(), done.data_ptr(), stream)

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    sharding = importlib.import_module("q-learning_b200.sharding")

    def reduce_stats():
        """episode-stat reduction, off the step path: sum {return, episodes, steps}, max {-min, max} over ranks (NCCL)."""
        env.stats_export(stats_vec.data_ptr(), stream)
        return sharding.reduce_episode_stats(stats_vec, dist if distributed else None)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        launch()
    torch.cuda.synchronize()
    # a few launches are ~1 ms: keep warming (untimed) until clocks have settled. A fixed count of launches, not a fixed time, so that
    # the timed launches start from the same env state in every run and on every build, and compute the same outputs (--dump-outputs).
    for _ in range(SETTLE_LAUNCHES):
        launch()
    torch.cuda.synchronize()
    reduce_stats()
    # ---- timed region: exactly K launches, device resident inputs ----
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        launch()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if distributed:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, q, torch, env, reward, done, dev, stream)
    # keep the GPU loaded for the clock sampler if the timed region was short (untimed, same launches)
    t_load = time.time()
    while sampler and time.time() - t_load < 1.0:
        for _ in range(20):
            launch()
        torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    stats = reduce_stats()

    units_per_step = n_envs * k_inner * world
    value = units_per_step * args.steps / (ms * 1e-3)

    # ---- e2e: the same metric through the host-buffer C-ABI call (pinned staging, H2D actions, D2H reward+done) ----
    # Every step copies that step's actions host->device from page-locked memory and reads reward + done back.
    pa, pr, pd = q.PinnedArray((k_inner, n_envs), np.uint8), q.PinnedArray((k_inner, n_envs), np.float32), q.PinnedArray((k_inner, n_envs), np.uint8)
    pa.array[:] = actions.cpu().numpy()
    a_host, r_host, d_host = pa.array, pr.array, pd.array
    e2e_steps = max(3, min(args.steps, 50))
    for _ in range(3):
        env.step_many(a_host, out=(r_host, d_host))
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        env.step_many(a_host, out=(r_host, d_host))
    torch.cuda.synchronize()
    dt_sync = time.perf_counter() - t0
    # pipelined form (qlc_env_step_host_submit / _wait): the synthetic action stream does not depend on earlier results, so
    # step k+1 is validated and queued while step k runs; two page-locked buffer sets, every step's result waited for and read on the host
    pa2, pr2, pd2 = q.PinnedArray((k_inner, n_envs), np.uint8), q.PinnedArray((k_inner, n_envs), np.float32), q.PinnedArray((k_inner, n_envs), np.uint8)
    pa2.array[:] = pa.array
    sets = ((pa.array, pr.array, pd.array), (pa2.array, pr2.array, pd2.array))
    e2e_check = 0.0
    for i in range(4):
        env.step_many_submit(*sets[i & 1])
    env.step_many_wait()
    barrier()
    t0 = time.perf_counter()
    env.step_many_submit(*sets[0])
    for i in range(1, e2e_steps):
        env.step_many_submit(*sets[i & 1])           # queue step i (its buffer set was consumed after step i-2) ...
        env.step_many_wait(1)                        # ... then wait for step i-1 and consume its read-back result on the host
        prev = sets[(i - 1) & 1]
        e2e_check += float(prev[1][k_inner - 1, n_envs - 1]) + float(prev[2][0, 0])
    env.step_many_wait()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if distributed:
        t = torch.tensor([dt, dt_sync], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt, dt_sync = float(t[0].item()), float(t[1].item())
    e2e_value = units_per_step * e2e_steps / dt
    e2e_bytes = (int(a_host.nbytes), int(r_host.nbytes + d_host.nbytes))
    e2e_check += float(r_host.sum()) + float(pr2.array.sum())          # the read-back results are consumed on the host
    e2e_sync_value = units_per_step * e2e_steps / dt_sync

    stats_every_step = None if args.no_extra else measure_stats_reduce_every_step(q, torch, dist if distributed else None, env, launch, stream, rank, world, dev, barrier, args.steps)
    replay = None if args.no_extra else measure_replay_sampling(q, torch, dist if distributed else None, rb, dev, stream, world, barrier)
    loops = {} if args.no_extra else measure_actor_loops(q, torch, dist if distributed else None, env, rb, dev, stream, world, barrier)
    if not args.no_extra and not args.no_learner:
        loops.update(measure_actor_loop_learner(torch, dist if distributed else None, rank, local_rank, world, dev, barrier, n_envs))
    extra = {}
    cpu_baseline = None
    if rank == 0:
        peak, peak_src = _peaks()
        launch_ms = ms / args.steps
        achieved = launch_bytes(n_envs, k_inner) / (launch_ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": "env_advance_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "peak_source": peak_src, "frac_of_nominal_8tbs": achieved / 8000.0,   # north_star quotes the ~8 TB/s datasheet figure
                    "traffic": _ncu_traffic("env_advance_kernel"),
                    "algorithmic_bytes_per_launch": launch_bytes(n_envs, k_inner),
                    "algorithmic_bytes_formula": "7066 B x envs x steps_per_launch + 106 B x envs (state read + written once per launch)"}
        if not args.no_extra:
            extra = measure_extras(q, torch, env, rb, dev, stream, peak, replay, cpu_baseline=(world == 1 and not args.no_cpu_baseline))
        if world == 1 and not args.no_cpu_baseline:
            from oracle import oracle as O
            O.build()
            cores = os.cpu_count() or 1
            s_envs, s_steps = n_envs, min(k_inner, 64)
            O.bench_env_steps(s_envs, 2, SEED, cores)                       # page in, spin up the thread pool (untimed)
            s_reps, secs = 0, 0.0
            while s_reps < 2 or (secs * cores < 16.0 and s_reps < 64):       # about 16+ core-seconds of CPU work, whole bench steps
                secs += O.bench_env_steps(s_envs, s_steps, SEED + s_reps, cores)
                s_reps += 1
            cpu_baseline = {"value": s_reps * s_envs * s_steps / secs, "unit": "env-steps/s", "cores": cores, "kind": "port",
                            "sample": "%d bench steps on the CPU oracle: each %d envs x %d env-steps, %d OpenMP threads, %.1f s wall (%.0f core-seconds)" % (s_reps, s_envs, s_steps, cores, secs, secs * cores)}
        line = {
            "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": _config(n_envs, k_inner, args.replay_capacity, world),
            "roofline": roofline, "cpu_baseline": cpu_baseline, "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": e2e_bytes[0], "d2h_bytes_per_step": e2e_bytes[1],
                    "timing": "perf_counter around %d pipelined host-buffer C-ABI steps (qlc_env_step_host_submit per step, two page-locked buffer sets, qlc_env_step_host_wait(1) + a host read of the previous step's result per step), max over ranks" % e2e_steps,
                    "synchronous_call": {"value": e2e_sync_value, "unit": "env-steps/s", "note": "qlc_env_step_host: submit + wait per step (what a caller whose next actions depend on the result uses)"},
                    "result_checksum": e2e_check},
            "gpu_launches": args.steps,
            "library": dict(build, note="profiling=0: release build, QLC_DEBUG_SKIP is compiled out; src_hash = sha256 of the sources the binary was built from"),
            "episode_stats": dict(stats, reduced_with="nccl all_reduce (2 tiny calls, off the step path)" if distributed else "single rank"),
            "env_error_flags": env.error_flags(),
            "env_error_flags_note": "OR of the sticky per-env flags after all launches of this run (1 wall-distance assert, 2 approximation range, 4 reflection bound, "
                                    "8 bisection bound, 16 degenerate contact, 32 bad action, 64 hand-over time-out): states in which the reference panics or "
                                    "recurses without bound (mechanics.rs:265,284,303,361-389,511); %d of %d envs flagged on rank 0; the oracle raises the same flags "
                                    "on the same steps (test_rare_events_parity, test_soak)" % (int((env.read_state()["err"] != 0).sum()), n_envs),
        }
        line.update(extra)
        line.update(loops)
        if stats_every_step:
            line["stats_reduce_every_step"] = stats_every_step
        print(json.dumps(line), flush=True)
    env.close()
    if distributed:
        dist.barrier()
        dist.destroy_process_group()


def dump_outputs(out_dir, q, torch, env, reward, done, dev, stream):
    """--dump-outputs DIR: what the last timed launch handed its caller, as DIR/<name>.npy in f32 / f64, so that two builds run with
    the same arguments can be compared output for output: reward and done [steps_per_launch][envs], the env state it advanced to
    (one file per field, u32 fields as f64, the 64-bit brick masks as two f64 halves) and the 4-frame observation stacks
    [envs][slot][y][x] of the first DUMP_OBS_ENVS of those envs. Beyond 4,096 envs, or 32 MiB of per-env arrays, the envs are a
    fixed seeded sample, so the files stay under 64 MB together (at most 32 MiB + 28.9 MB of stacks). Rank 0's shard only."""
    n, k = env.n_envs, reward.shape[0]
    st = env.read_state()
    state = {name: st[name] for name in ("ball_cx", "ball_cy", "ball_dx", "ball_dy", "pad_min_x", "pad_max_x", "pad_speed")}
    state.update({name: st[name].astype(np.float64) for name in ("score", "episode_step", "episode", "err")})
    state["finished"] = st["finished"].astype(np.float32)
    state["bricks_lo"] = (st["bricks"] & np.uint64(0xFFFFFFFF)).astype(np.float64)
    state["bricks_hi"] = (st["bricks"] >> np.uint64(32)).astype(np.float64)
    per_env = 2 * 4 * k + sum(a.itemsize for a in state.values())
    keep = max(1, min(n, 4096, (32 << 20) // per_env))
    ids = np.arange(n) if keep == n else np.sort(np.random.default_rng(SEED).choice(n, keep, replace=False))
    obs = torch.empty((n, 4, 84, 84), dtype=torch.uint8, device=dev)
    env.obs_device(q.LAYOUT_U8_BHYX, obs.data_ptr(), stream)
    out = {"reward": reward.cpu().numpy()[:, ids], "done": done.cpu().numpy()[:, ids].astype(np.float32),
           "obs": obs[torch.from_numpy(ids[:DUMP_OBS_ENVS]).to(dev)].float().cpu().numpy()}
    out.update(("state_" + name, a[ids]) for name, a in state.items())
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def measure_stats_reduce_every_step(q, torch, dist, env, launch, stream, rank, world, dev, barrier, steps):
    """The episode-stat reduction THROUGH THE C ABI (qlc_comm_init: NCCL bound by dlopen inside libqlcuda.so; one ncclAllGather of
    5 doubles + a combine kernel on the communicator's low-priority side stream) enqueued after EVERY bench step, against the
    same launches without it: it must not be on the step path. The 128-byte NCCL id travels over the host's own channel
    (here torch.distributed broadcast; a Rust host would use a file or a socket)."""
    steps = max(20, min(steps, 300))

    def timed(with_reduce):
        for _ in range(5):
            launch()
            if with_reduce:
                env.stats_allreduce(stream)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            launch()
            if with_reduce:
                env.stats_allreduce(stream)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1) / steps
        if dist is not None:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    ms_without = timed(False)
    if dist is not None:
        ident = [q.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ident, src=0)
        env.comm_init(rank, world, ident[0])
    else:
        env.comm_init(0, 1, q.comm_unique_id())            # a real one-rank NCCL communicator
    ms_with = timed(True)
    ms_without2 = timed(False)
    env.stats_allreduce(stream)
    g = env.stats_global(wait=True)
    local = env.stats()
    info = env.comm_info()
    if dist is not None:                                    # cross-check against torch.distributed's own reduction
        t = torch.tensor([local["sum_return"], local["episodes"], local["steps"]], dtype=torch.float64, device=dev)
        dist.all_reduce(t)
        ok = [int(x) for x in t.tolist()] == [g["sum_return"], g["episodes"], g["steps"]]
    else:
        ok = g == local
    return {"ms_per_step_with": ms_with, "ms_per_step_without": min(ms_without, ms_without2), "ms_per_step_without_before_after": [ms_without, ms_without2],
            "overhead_frac": ms_with / min(ms_without, ms_without2) - 1.0, "steps": steps, "nccl_version": info["nccl_version"], "nccl_ranks": info["nccl_ranks"],
            "world": world, "matches_torch_distributed": bool(ok), "global": g,
            "note": "qlc_stats_allreduce after every bench step (C ABI; NCCL via dlopen; side stream, snapshot taken by the step kernel's last CTA), max over ranks"}


def measure_actor_loops(q, torch, dist, env, rb, dev, stream, world, barrier):
    """BASELINE configs[4] without the (out-of-scope) learner, on EVERY rank (env + replay shards, no data-path collective),
    device-timed, max over ranks:
    (1) actor_loop: per iteration a fresh action batch from a device-side policy stand-in (uniform random, like the learner's
        first 50k steps), ONE env-step launch, and on every 4th step (the learner's gate, self_driving_tf_q_learner.rs:181) a
        distinct-index sample + f32 [32,84,84,4] s/s' gather;
    (2) actor_loop_qnet: the same with the greedy action of the tcgen05 Q-network forward over all envs (closed loop on the GPU)."""
    per = 4 * 84 * 84
    n = env.n_envs
    idx = torch.empty((32,), dtype=torch.int32, device=dev)
    st = torch.empty((32, per), dtype=torch.float32, device=dev); nx = torch.empty((32, per), dtype=torch.float32, device=dev)
    r = torch.empty((32,), dtype=torch.float32, device=dev); a = torch.empty((32,), dtype=torch.uint8, device=dev); d = torch.empty((32,), dtype=torch.uint8, device=dev)
    rew1 = torch.empty((1, n), dtype=torch.float32, device=dev); done1 = torch.empty((1, n), dtype=torch.uint8, device=dev)
    acts = torch.empty((1, n), dtype=torch.uint8, device=dev)
    net = q.QNetwork(env, _random_qnet_weights(q))

    def sample_every_4th(i):
        if rb.should_sample(i, rb.len(), 32):              # ONE launch: the gather kernel draws the distinct indices itself
            rb.sample_gather_device(32, 1, i, q.LAYOUT_F32_BXYH, idx.data_ptr(), st.data_ptr(), nx.data_ptr(), r.data_ptr(), a.data_ptr(), d.data_ptr(), stream)

    def iter_random(i):                       # the learner's pure-random phase: the step kernel draws the actions itself (qlc_env_step_random)
        env.step_random_device(1, acts.data_ptr(), rew1.data_ptr(), done1.data_ptr(), stream)
        sample_every_4th(i)

    def iter_torch_policy(i):                 # a policy stand-in outside the library: one more kernel (and its host dispatch) per iteration
        ra = torch.randint(0, 3, (1, n), dtype=torch.uint8, device=dev)
        env.step_device(ra.data_ptr(), 1, rew1.data_ptr(), done1.data_ptr(), stream)
        sample_every_4th(i)

    def iter_qnet(i):
        net.forward_device(None, n, 0, None, acts.data_ptr(), None, stream)                      # predict_action for every env
        env.step_device(acts.data_ptr(), 1, rew1.data_ptr(), done1.data_ptr(), stream)
        sample_every_4th(i)

    res = []
    for fn, iters in ((iter_random, 400), (iter_qnet, 200), (iter_torch_policy, 400)):
        for i in range(8):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            fn(i)
        e1.record()
        barrier()
        res.append(e0.elapsed_time(e1) / iters)
    net.close()
    if world > 1:
        t = torch.tensor(res, dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res = [float(x) for x in t.tolist()]
    scope = "%d GPU(s), %d envs each, slowest rank" % (world, n)
    return {
        "actor_loop": {"env_steps_per_sec": world * n / (res[0] * 1e-3), "minibatches_per_sec": world * 0.25 / (res[0] * 1e-3), "us_per_iteration": res[0] * 1e3, "n_gpus": world,
                       "kernels_per_iteration": 1.25,
                       "note": "1 step launch per iteration with the uniform random policy of the learner's pure-random phase drawn inside the step kernel "
                               "(qlc_env_step_random; actions, reward, done written out), one-launch sample+gather B=32 f32 every 4th step; no learner; " + scope},
        "actor_loop_torch_policy": {"env_steps_per_sec": world * n / (res[2] * 1e-3), "us_per_iteration": res[2] * 1e3, "kernels_per_iteration": 2.25,
                                    "note": "same with the actions from torch.randint (r01's actor_loop): the extra kernel's host dispatch (~7 us) bounds the iteration"},
        "actor_loop_qnet": {"env_steps_per_sec": world * n / (res[1] * 1e-3), "minibatches_per_sec": world * 0.25 / (res[1] * 1e-3), "us_per_iteration": res[1] * 1e3, "n_gpus": world,
                            "qnet_tflops_per_gpu": QNET_FLOP_PER_OBS * n / (res[1] * 1e-3) / 1e12,
                            "note": "closed loop on the GPU: Q-network forward (greedy action for all envs) -> 1 env-step launch -> sample+gather B=32 f32 every 4th step; no learner; " + scope},
    }


def measure_actor_loop_learner(torch, dist, rank, local_rank, world, dev, barrier, n_envs):
    """BASELINE configs[4] WITH a learner attached, on every rank: the vectorised DQN loop of examples/dqn_breakout_torch.py — env
    shard + replay shard on the GPU (this repo), zero-copy one-launch sample+gather into the tensors of a device-resident torch
    Q-network of the reference architecture (library code, the stand-in for the reference's TensorFlow model: forward for the
    greedy actions and the TD target, forward + backward + Adam for every minibatch), one minibatch of 32 per 4 env-steps like
    the reference (self_driving_tf_q_learner.rs:181). Run twice: with the model, and with the model calls skipped (the data path
    alone), which attributes the iteration time. No collective on the path (each rank trains its own replica here; a real
    multi-GPU learner would all-reduce gradients - the learner is outside this repo's scope)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("dqn_breakout_torch", os.path.join(ROOT, "examples", "dqn_breakout_torch.py"))
    ex = importlib.util.module_from_spec(spec); spec.loader.exec_module(ex)
    iters = 12
    res = []
    for skip in (False, True):
        ex.run(n_envs, 2, quiet=True, device=local_rank, env_id_base=rank * n_envs, seed=SEED, skip_model=skip, random_phase_steps=0)   # warm-up (cudnn autotune, allocator)
        barrier()
        t0 = time.perf_counter()
        out = ex.run(n_envs, iters, quiet=True, device=local_rank, env_id_base=rank * n_envs, seed=SEED, skip_model=skip, random_phase_steps=0)
        torch.cuda.synchronize()
        res.append(out["seconds"])
    secs_full, secs_data = res
    if dist is not None:
        t = torch.tensor([secs_full, secs_data], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        secs_full, secs_data = float(t[0].item()), float(t[1].item())
    steps = n_envs * iters
    return {"actor_loop_learner": {
        "env_steps_per_sec": world * steps / secs_full, "minibatches_per_sec": world * (steps // 4) / secs_full, "ms_per_iteration": 1e3 * secs_full / iters,
        "data_path_only_ms_per_iteration": 1e3 * secs_data / iters, "learner_share_of_iteration": 1.0 - secs_data / secs_full, "n_gpus": world,
        "bound_by": "the torch model (forward + backward + Adam on %d samples and two forwards per iteration); the env step, replay insert and the one-launch "
                    "sample+gather of an iteration are the data_path_only time" % (n_envs // 4 * 32),
        "note": "%d envs per GPU, %d iterations, greedy actions from the model on every iteration (no pure-random phase), wall clock incl. env creation "
                "excluded; slowest rank; compare actor_loop_cpu_baseline (the restated reference data path, 1 env, 1 thread, no model)" % (n_envs, iters)}}


def measure_replay_sampling(q, torch, dist, rb, dev, stream, world, barrier):
    """BASELINE configs[2] on EVERY rank (one replay shard per GPU, no cross-GPU gather): Philox distinct-index sample + gather of
    the s and s' frame stacks into device buffers in ONE kernel launch (the gather kernel derives the indices), u8 [b][slot][y][x]
    and the reference's f32 [b][x][y][slot]; device-timed, max over ranks, whole-job transitions/s. The gather with GIVEN indices
    (get_many; those of the last call) is timed beside it; 8,192 transitions read 289 MB of frames > L2."""
    per = 4 * 84 * 84
    keys, times = [], []
    for batch, n_batches in ((32, 1), (512, 1), (32, 256), (512, 16)):
        for layout, name, bps, dt in ((q.LAYOUT_U8_BHYX, "u8", BYTES_PER_SAMPLE_U8, torch.uint8), (q.LAYOUT_F32_BXYH, "f32", BYTES_PER_SAMPLE_F32, torch.float32)):
            n = batch * n_batches
            idx = torch.empty((n,), dtype=torch.int32, device=dev)
            st = torch.empty((n, per), dtype=dt, device=dev); nx = torch.empty((n, per), dtype=dt, device=dev)
            r = torch.empty((n,), dtype=torch.float32, device=dev); a = torch.empty((n,), dtype=torch.uint8, device=dev); d = torch.empty((n,), dtype=torch.uint8, device=dev)

            def gather():
                rb.gather_device(idx.data_ptr(), n, layout, st.data_ptr(), nx.data_ptr(), r.data_ptr(), a.data_ptr(), d.data_ptr(), stream)

            def once(c):                                   # sample + gather: ONE kernel launch
                rb.sample_gather_device(batch, n_batches, c, layout, idx.data_ptr(), st.data_ptr(), nx.data_ptr(), r.data_ptr(), a.data_ptr(), d.data_ptr(), stream)
            for c in range(3):
                once(c)
            reps = 30
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            e0.record()
            for c in range(reps):
                once(10 + c)
            e1.record()
            barrier()
            ms = e0.elapsed_time(e1) / reps
            e0.record()
            for c in range(reps):
                gather()
            e1.record()
            barrier()
            ms_g = e0.elapsed_time(e1) / reps
            ms_p = 0.0
            keys.append((batch, n_batches, name, bps, n))
            times += [ms, ms_g, ms_p]
            del idx, st, nx
    # end to end through the reference-facing host calls, in the reference's call pattern: the learner draws the ids itself on the
    # host (its private generate_distinct_random_ids, self_driving_tf_q_learner.rs:183,276-296), then get_many +
    # batch_to_multi_dim_array for state_next and state into page-locked host arrays the caller reads. f32 stacks cross PCIe as u8
    # (1/4 of the bytes) and are widened into the caller's arrays by the library's host pool.
    host_keys, host_check = [], 0.0
    host_rng = np.random.default_rng(SEED)
    for batch in (32, 512):
        for layout, name, isz in ((q.LAYOUT_U8_BHYX, "u8", 1), (q.LAYOUT_F32_BXYH, "f32", 4)):
            for c in range(3):
                rb.get_many(host_rng.choice(rb.len(), size=batch, replace=False).astype(np.uint32), layout, reuse=True)
            reps = 20
            id_lists = [host_rng.choice(rb.len(), size=batch, replace=False).astype(np.uint32) for _ in range(reps)]   # the learner's own draw, not this repo's code
            barrier()
            t0 = time.perf_counter()
            for c in range(reps):
                g = rb.get_many(id_lists[c], layout, reuse=True)
                host_check += float(g.reward.sum()) + float(g.state_next[batch - 1].ravel()[-1])
            times.append((time.perf_counter() - t0) / reps * 1e3)
            host_keys.append((batch, name, batch * (2 * per + 4 + 1 + 1), batch * 2 * per * isz))
    if world > 1:
        t = torch.tensor(times, dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        times = [float(x) for x in t.tolist()]
    peak, _ = _peaks()
    res = {}
    e2e_host = {}
    for i, (batch, name, d2h, host_bytes) in enumerate(host_keys):
        ms = times[3 * len(keys) + i]
        e2e_host["batch%d_%s" % (batch, name)] = {"transitions_per_sec": world * batch / (ms * 1e-3), "ms_per_minibatch": ms, "d2h_bytes_per_minibatch": d2h,
                                                   "host_tensor_bytes_per_minibatch": host_bytes, "host_tensor_gbs_per_gpu": host_bytes / (ms * 1e-3) / 1e9}
    for i, (batch, n_batches, name, bps, n) in enumerate(keys):
        ms, ms_g, ms_p = times[3 * i], times[3 * i + 1], times[3 * i + 2]
        rate = n / (ms * 1e-3)                       # per GPU, slowest rank
        res["batch%d_x%d_%s" % (batch, n_batches, name)] = {
            "transitions_per_sec": world * rate, "ms_per_call": ms, "achieved_gbs_per_gpu": rate * bps / 1e9, "frac_of_peak": rate * bps / 1e9 / peak,
            "frac_of_nominal_8tbs": rate * bps / 1e9 / 8000.0, "bytes_per_transition": bps, "kernels_per_call": 1,
            "gather_kernel_alone": {"ms_per_launch": ms_g, "achieved_gbs_per_gpu": n * bps / (ms_g * 1e-3) / 1e9, "frac_of_peak": n * bps / (ms_g * 1e-3) / 1e9 / peak}}
        if ms_p > 0.0:
            res["batch%d_x%d_%s" % (batch, n_batches, name)]["sample_prefetched_on_second_stream"] = {
                "transitions_per_sec": world * n / (ms_p * 1e-3), "ms_per_call": ms_p, "frac_of_peak": n * bps / (ms_p * 1e-3) / 1e9 / peak}
    return {"metric": "sampled_transitions_per_sec", "n_gpus": world, "replay_len_per_gpu": rb.len(), "results": res,
            "e2e_host": dict(e2e_host, timing="perf_counter around ReplayBuffer.get_many(reuse=True) per minibatch with host-drawn distinct ids (drawn before the timed loop; host index array in, "
                                              "page-locked host stacks out, read on the host), max over ranks; stacks cross PCIe as u8, f32 ones are widened by %d host threads" % _host_threads(),
                             result_checksum=host_check),
            "note": "qlc_replay_sample_gather: Philox distinct ids drawn inside the gather kernel + s and s' stacks, ONE launch per call, device buffers, every rank on its own replay shard, max over ranks; "
                    "transitions_per_sec is the whole job, GB/s and fractions are per GPU; minibatches per call = the x factor"}


def _host_threads():
    n = os.environ.get("QLC_HOST_THREADS")
    if n and int(n) > 0:
        return int(n)
    ranks = int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1)
    return max(1, min(16, (os.cpu_count() or 2) // max(ranks, 1)))


def measure_extras(q, torch, env, rb, dev, stream, peak, replay, cpu_baseline=True):
    """Secondary numbers in the same run (rank 0): the CPU baseline of the replay path and the 65,536-env shard (configs[3])."""
    out = {"replay_sample": replay}
    if cpu_baseline:
        # the reference's learn_episode data path without the model (one env, one thread, like the reference learner): step_as_rc +
        # ReplayBuffer::add + every 4th step sample 32 + tensorise state and state_next
        from oracle import oracle as O
        a_steps = 12000                                         # about 5 s of single-thread CPU work
        a_secs = O.bench_actor_loop(a_steps, 4096, 32, SEED)
        out["actor_loop_cpu_baseline"] = {"value": a_steps / a_secs, "unit": "env-steps/s", "minibatches_per_sec": 0.25 * a_steps / a_secs, "cores": 1, "kind": "port",
                                          "sample": "%d env-steps of one env: step+render+grayscale+ring+state clone+replay add, every 4th step sample 32 distinct + f32 tensorisation of state and state_next (no model), CPU oracle, 1 thread, %.1f s" % (a_steps, a_secs)}
        # the reference's replay path on the host (ReplayBuffer::get_many + batch_to_multi_dim_array for state and state_next,
        # generate_distinct_random_ids), single-threaded like the reference learner; bounded sample
        from oracle import oracle as O
        s_envs, s_cap, s_batch, s_nb = 64, 4096, 32, 8000     # about 10 s of single-thread CPU work
        secs = O.bench_sample(s_envs, s_cap, s_batch, s_nb, SEED)
        out["replay_sample"]["cpu_baseline"] = {"value": s_batch * s_nb / secs, "unit": "sampled transitions/s", "cores": 1, "kind": "port",
                                                "sample": "%d minibatches of %d (f32 [b][x][y][slot] state + state_next) from a %d-transition replay of %d envs, CPU oracle, 1 thread, %.1f s" % (s_nb, s_batch, s_cap, s_envs, secs)}
    # 65,536 envs on this GPU (configs[3] shard size), 16 env-steps per launch
    try:
        big = q.BreakoutEnvironment(n_envs=65536, seed=SEED + 1, replay_capacity=65536 * 32, device=dev.index)
        k = 16
        acts = torch.randint(0, 3, (k, 65536), dtype=torch.uint8, device=dev)
        for _ in range(3):
            big.step_device(acts.data_ptr(), k, None, None, stream)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 20
        e0.record()
        for _ in range(reps):
            big.step_device(acts.data_ptr(), k, None, None, stream)
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        rate = 65536 * k / (ms * 1e-3)
        out["envs_65536"] = {"env_steps_per_sec": rate, "ms_per_launch": ms, "steps_per_launch": k, "achieved_gbs": launch_bytes(65536, k) / (ms * 1e-3) / 1e9,
                             "frac_of_peak": launch_bytes(65536, k) / (ms * 1e-3) / 1e9 / peak}
        for _ in range(3):
            big.step_device(acts.data_ptr(), 1, None, None, stream)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(100):
            big.step_device(acts.data_ptr(), 1, None, None, stream)
        e1.record(); torch.cuda.synchronize()
        ms1 = e0.elapsed_time(e1) / 100
        out["envs_65536"]["single_step_launch"] = {"env_steps_per_sec": 65536 / (ms1 * 1e-3), "us_per_launch": ms1 * 1e3}
        # closed actor loop on the big shard: Q-network forward for all 65,536 envs -> one env-step launch
        net = q.QNetwork(big, _random_qnet_weights(q))
        acts1 = torch.empty((1, 65536), dtype=torch.uint8, device=dev)
        for _ in range(3):
            net.forward_device(None, 65536, 0, None, acts1.data_ptr(), None, stream)
            big.step_device(acts1.data_ptr(), 1, None, None, stream)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(20):
            net.forward_device(None, 65536, 0, None, acts1.data_ptr(), None, stream)
            big.step_device(acts1.data_ptr(), 1, None, None, stream)
        e1.record(); torch.cuda.synchronize()
        ms2 = e0.elapsed_time(e1) / 20
        out["envs_65536"]["actor_loop_qnet"] = {"env_steps_per_sec": 65536 / (ms2 * 1e-3), "ms_per_iteration": ms2,
                                                "qnet_tflops": QNET_FLOP_PER_OBS * 65536 / (ms2 * 1e-3) / 1e12,
                                                "note": "Q-network forward (greedy action for every env) + 1 env-step launch per iteration"}
        net.close()
        big.close()
    except Exception as ex:  # e.g. not enough free HBM next to the main shard
        out["envs_65536"] = {"error": str(ex)}
    # one env-step per launch (the learner-driven mode: actions depend on the previous state)
    acts1 = torch.randint(0, 3, (1, env.n_envs), dtype=torch.uint8, device=dev)
    for _ in range(10):
        env.step_device(acts1.data_ptr(), 1, None, None, stream)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(500):
        env.step_device(acts1.data_ptr(), 1, None, None, stream)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 500
    out["single_step_launch"] = {"env_steps_per_sec": env.n_envs / (ms * 1e-3), "us_per_launch": ms * 1e3}
    out.update(measure_qnet(q, torch, env, dev, stream))
    # the same drop-in calls from a COMPILED host (plain C against include/ql_cuda.h - what a Rust ql-cuda crate pays), without
    # ctypes and numpy around them: its own process, its own env handles
    try:
        exe = q._build.build_c_host_tool()
        if exe:
            r = subprocess.run([exe, "--json"], capture_output=True, text=True, timeout=120)
            if r.returncode == 0:
                out["compiled_host_calls"] = dict(json.loads(r.stdout.strip().splitlines()[-1]),
                                                  note="tools/cabi/c_abi_latency.c (C, gcc -O2) through the C ABI: one env stepped one call at a time; one state handle -> f32 tensor; "
                                                       "qlc_replay_gather_host of a minibatch into page-locked host tensors on a 4,096-env shard with a 1 M ring; microseconds per call")
            else:
                out["compiled_host_calls"] = {"error": (r.stderr or r.stdout)[-300:]}
    except Exception as ex:
        out["compiled_host_calls"] = {"error": str(ex)}
    return out




def _tensor_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["bf16_tflops"]), "measured (MEASURED_PEAKS.json bf16_tflops, burst)"
    except Exception:
        return 2250.0, "nominal dense bf16"


def _random_qnet_weights(q, seed=7):
    """random-init weights of the reference architecture (glorot-uniform kernels like Keras, zero biases)"""
    rng = np.random.default_rng(seed)
    w = {}
    for name, shape in q.QNET_SHAPES.items():
        if name.endswith("kernel"):
            lim = np.sqrt(6.0 / (int(np.prod(shape[:-1])) + shape[-1]))
            w[name] = rng.uniform(-lim, lim, size=shape).astype(np.float32)
        else:
            w[name] = np.zeros(shape, dtype=np.float32)
    return w


def measure_qnet(q, torch, env, dev, stream):
    """SURVEY.md 8f-3: the Q-network forward on tcgen05 (predict_action for every env, straight from the frame ring).
    Random-init weights of the reference architecture (no checkpoints here)."""
    out = {}
    w = _random_qnet_weights(q)
    net = q.QNetwork(env, w)
    n = env.n_envs
    acts = torch.empty((1, n), dtype=torch.uint8, device=dev)
    qv = torch.empty((n, 3), dtype=torch.float32, device=dev)
    for _ in range(5):
        net.forward_device(None, n, 0, qv.data_ptr(), acts.data_ptr(), None, stream)
    torch.cuda.synchronize()
    reps = 50
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        net.forward_device(None, n, 0, qv.data_ptr(), acts.data_ptr(), None, stream)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    peak, src = _tensor_peak()
    tf = QNET_FLOP_PER_OBS * n / (ms * 1e-3) / 1e12
    # how often the bf16 tensor-core path picks the action a plain fp32 forward of the same Keras model picks - ALL envs, ties and
    # near-ties included (library code, outside every timed region; TF32 off)
    agree = None
    try:
        tio = importlib.import_module("q-learning_b200.torch_io")
        F = torch.nn.functional
        old_flags = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
        torch.backends.cudnn.allow_tf32 = False; torch.backends.cuda.matmul.allow_tf32 = False
        x = tio.observe(env, q.LAYOUT_F32_BXYH).permute(0, 3, 1, 2).contiguous()       # NCHW with H = x, W = y
        for i, stride in ((1, 4), (2, 2), (3, 1)):
            k = torch.from_numpy(w["conv%d_kernel" % i]).to(dev).permute(3, 2, 0, 1).contiguous()
            x = torch.relu(F.conv2d(x, k, torch.from_numpy(w["conv%d_bias" % i]).to(dev), stride=stride))
        x = x.permute(0, 2, 3, 1).reshape(n, -1)
        x = torch.relu(x @ torch.from_numpy(w["dense1_kernel"]).to(dev) + torch.from_numpy(w["dense1_bias"]).to(dev))
        ref = x @ torch.from_numpy(w["dense2_kernel"]).to(dev) + torch.from_numpy(w["dense2_bias"]).to(dev)
        torch.cuda.synchronize()
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old_flags
        scale = float(ref.abs().max())
        srt = ref.sort(dim=1).values
        gap = (srt[:, 2] - srt[:, 1]) / max(scale, 1e-30)
        same = ref.argmax(dim=1).to(torch.uint8) == acts[0]
        agree = {"fraction_of_envs_with_the_fp32_greedy_action": float(same.float().mean()), "envs": n,
                 "max_abs_q_error_over_max_abs_q": float((qv - ref).abs().max()) / max(scale, 1e-30),
                 "fraction_where_top2_gap_exceeds_1e-2_of_max_abs_q": float((gap > 1e-2).float().mean()),
                 "agreement_among_those": float(same[gap > 1e-2].float().mean()) if bool((gap > 1e-2).any()) else None,
                 "note": "fp32 torch forward of the same random-init Keras model on the current observation of every env (cuDNN / cuBLAS, TF32 off) against "
                         "the bf16-operand tcgen05 path; disagreements are near-ties (top-2 Q gap below the bf16 error)"}
    except Exception as ex:   # a reporting extra must not take the bench line down
        agree = {"error": str(ex)}
    out["qnet_forward"] = {"observations_per_sec": n / (ms * 1e-3), "ms_per_forward": ms, "batch": n, "dtype": "bf16 operands, f32 accumulate (TMEM)",
                           "greedy_action_vs_fp32": agree,
                           "roofline": {"bound": "tensor", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak, "peak_source": src,
                                        "note": "convs are shifted-window implicit GEMMs with N = 32/64: bound by the 128 B/clk shared-memory operand fetch "
                                                "(40/48 cycles per MMA measured, tools/microbench/mma_rate.cu), not by the tensor pipe"},
                           "kernels_per_forward": 4}
    net.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)     # SURVEY.md 8(d): CUDA-event time over >= 1,000 launches after warm-up
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU, help="envs per GPU")
    ap.add_argument("--steps-per-launch", type=int, default=STEPS_PER_LAUNCH)
    ap.add_argument("--replay-capacity", type=int, default=REPLAY_CAPACITY)
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary measurements")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-learner", action="store_true", help="skip the learner-in-the-loop section (profiling runs: it is thousands of library kernels)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (f32 / f64, under 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("bench.py: --gpus %d needs torchrun (one rank per GPU)" % args.gpus)
    run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
