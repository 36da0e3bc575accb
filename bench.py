#!/usr/bin/env python
"""bench.py — env-steps/sec of the B200 Procgen hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--game coinrun] ...

A "step" = one act()+observe() pass over one batch of `--envs-per-gpu` environments (default 65536,
BASELINE configs[1]: coinrun, distribution_mode=easy) with synthetic uniform-random actions.
  value   whole-job env-steps/s, actions already resident in HBM, observations left in HBM
  e2e     same metric through the libenv C ABI with HOST buffers (pinned): actions H2D and
          rgb/rew/first/info D2H inside the timed region — the drop-in path gym3's CEnv would drive
  roofline  HBM bound; algorithmic bytes = 12288 B rgb write per env-step (SURVEY §8d)
  cpu_baseline  oracle/_ref (reference game logic compiled unmodified + restated Qt raster) on the
          host cores, bounded sample
With --impl reference the reference's CPU implementation (oracle/_ref, all host threads) is timed
instead and reported on the same metric/config. --dump-outputs DIR saves what the last timed step
returned, so that two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

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

ALGO_BYTES_PER_ENV_STEP = 64 * 64 * 3  # SURVEY §8(d)
METRIC = "env-steps/sec"
CLOCK_WARM_ROUNDS = 20   # of 20 steps each, before the steady-state timed steps
DUMP_BYTES = 64 << 20    # --dump-outputs: all files together


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "25", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference_rate(game, mode, budget_s=15.0, envs_per_worker=64, workers=None):
    """Times oracle/_ref on ALL host cores on a bounded sample of the same workload.

    The reference scales across cores by running independent VecGames (its own thread pool is one
    mutex + notify_all per game and gets slower with threads for cheap steps, SURVEY §8d), so the
    baseline is `workers` = nproc independent reference VecGames (num_threads=0, 64 envs each),
    each driven by its own host thread (ctypes releases the GIL inside libenv_act/observe)."""
    import numpy as np

    from oracle.ref_env import RefVecEnv

    cores = host_cpu_info()["usable"]
    workers = cores if workers is None else workers
    n = envs_per_worker
    envs = [RefVecEnv(n, game, distribution_mode=mode, num_levels=0, start_level=0, rand_seed=w, num_threads=0)
            for w in range(workers)]
    counts = [0] * workers
    start = threading.Barrier(workers + 1)
    t_end = [0.0]

    def work(w):
        env = envs[w]
        rng = np.random.RandomState(w)
        acts = rng.randint(0, 15, size=(64, n)).astype(np.int32)
        env.observe()
        for i in range(2):
            env.act(acts[i])
            env.observe()
        start.wait()
        i = 0
        while time.perf_counter() < t_end[0]:
            env.act(acts[i & 63])
            env.observe()
            i += 1
        counts[w] = i

    threads = [threading.Thread(target=work, args=(w,)) for w in range(workers)]
    for t in threads:
        t.start()
    t_end[0] = time.perf_counter() + budget_s + 3600.0
    start.wait()
    t0 = time.perf_counter()
    t_end[0] = t0 + budget_s
    for t in threads:
        t.join()
    el = time.perf_counter() - t0
    for e in envs:
        e.close()
    total = n * sum(counts)
    return total / el, {"cores": workers, "sample": f"{workers} independent reference VecGames x {n} envs, {sum(counts)} "
                        f"vec-steps total in {el:.1f}s (num_threads=0 each, one host thread per VecGame)",
                        "seconds": el, "env_steps": total}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.perf_counter()
    per_step_budget = max(1.0, min(20.0, 120.0 / max(1, args.steps + args.warmup)))
    rates = []
    detail = None
    for _ in range(args.warmup):
        cpu_reference_rate(args.game, args.mode, budget_s=min(per_step_budget, 2.0))
    for _ in range(args.steps):
        r, detail = cpu_reference_rate(args.game, args.mode, budget_s=per_step_budget)
        rates.append(r)
    value = sum(rates) / len(rates)
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * args.envs_per_gpu * args.gpus / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+u8", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": detail["cores"], "kind": "reference",
                         "host": host_cpu_info(), "sample": detail["sample"] + " per bench step; reference game logic compiled unmodified, "
                                   "Qt raster restated on CPU (Qt itself is not installable here)"},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(out))


def workload_config(args):
    return {"workload": f"{args.game} distribution_mode={args.mode} num_envs={args.envs_per_gpu}/GPU num_levels=0 rand_seed=0, "
                        "uniform random actions", "envs_per_gpu": args.envs_per_gpu, "game": args.game,
            "distribution_mode": args.mode,
            "parallelism": f"env-sharded x{args.gpus}, " + ("rgb gathered to rank 0 every step (NCCL)" if getattr(args, "gather", False)
                                                               else "no per-step collective"),
            "l2": "per-step working set (12 KiB obs + env state per env x num_envs) exceeds the 126 MB L2; no explicit flush"}


def host_cpu_info():
    """What the CPU arm can really use: affinity mask and cgroup quota next to os.cpu_count()."""
    info = {"os_cpu_count": os.cpu_count()}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        info["affinity"] = None
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:
            continue
    info["cgroup_cpu_quota"] = quota
    usable = info["affinity"] or info["os_cpu_count"] or 1
    if quota:
        usable = max(1, min(usable, int(quota + 0.5)))
    info["usable"] = usable
    return info


def timed_rollout(env, actions, t0, K, barrier, gather=False, dist=None):
    """K steps through the public API (env.act / env.observe), CUDA events on the launching stream."""
    import torch

    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    T = actions.shape[0]
    barrier()
    ev0.record()
    for t in range(K):
        env.act(actions[(t0 + t) % T])
        rew, ob, first = env.observe()                           # aliases of HBM buffers; nothing to copy
        if gather and dist is not None:
            env.gather_observations(0)                           # the one collective of SURVEY §8e
    ev1.record()
    barrier()
    return ev0.elapsed_time(ev1)


def reset_fraction(env, actions, t0, steps):
    """Share of env-steps that ended an episode (observe() returned first=1), untimed pass."""
    import torch

    T = actions.shape[0]
    acc = torch.zeros((), device=actions.device, dtype=torch.float64)
    for t in range(steps):
        env.act(actions[(t0 + t) % T])
        rew, ob, first = env.observe()
        acc += first.sum()
    return float(acc.item()) / (steps * env.num)


def dump_outputs(env, out_dir):
    """Writes what observe() returned after the last timed step as float32 .npy files: rew.npy and
    first.npy for every env, and rgb.npy for a fixed seeded sample of envs whose indices are in
    rgb_envs.npy, sized so that the four files stay within DUMP_BYTES."""
    import numpy as np
    import torch

    rew, ob, first = env.observe()
    n = rew.shape[0]
    per_frame = 64 * 64 * 3 * 4 + 8   # float32 frame + its float64 index
    room = DUMP_BYTES - 8 * n - 4 * 4096   # rew, first and the .npy headers
    if room < per_frame:
        raise SystemExit(f"--dump-outputs: {n} envs do not fit in {DUMP_BYTES} bytes")
    k = min(n, room // per_frame)
    envs = np.arange(n) if k == n else np.sort(np.random.RandomState(0).choice(n, k, replace=False))
    rgb = ob["rgb"][torch.as_tensor(envs, device=ob["rgb"].device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "rew.npy"), rew.float().cpu().numpy())
    np.save(os.path.join(out_dir, "first.npy"), first.float().cpu().numpy())
    np.save(os.path.join(out_dir, "rgb.npy"), rgb.float().cpu().numpy())
    np.save(os.path.join(out_dir, "rgb_envs.npy"), envs.astype(np.float64))


def max_over_ranks(x, dist, dev):
    import torch

    if dist is None:
        return x
    t = torch.tensor([x], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def run_ours(args):
    import numpy as np
    import torch

    from procgen_b200 import ProcgenGym3Env

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(0)
    dev = torch.device("cuda", torch.cuda.current_device())
    n = args.envs_per_gpu
    K, W = args.steps, args.warmup

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    env = ProcgenGym3Env(n, args.game, distribution_mode=args.mode, num_levels=0, start_level=0, rand_seed=0,
                         shard=(rank, world) if world > 1 else None)
    if args.gather and dist is not None and not args.nccl_gather:
        env.enable_peer_gather(0)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    T = 256
    actions = torch.randint(0, 15, (T, n), device=dev, dtype=torch.int32, generator=gen)
    if args.chunks:
        env.set_launch_shape(chunks=args.chunks, serialize=False)   # profiling aid: fixed launch shape
    env.observe()
    torch.cuda.synchronize()

    # ---- cold: right after the synchronised initial reset (every env at step 0 of its first episode)
    for t in range(W):
        env.act(actions[t])
        env.observe()
    cold_ms = max_over_ranks(timed_rollout(env, actions, W, K, barrier), dist, dev)
    steps_done = W + K

    # ---- desynchronise: a rollout long enough that episode boundaries (level generation) are spread
    # over the steps the way they are in training; SURVEY §8(d) measures 1000 steps after 100 warm-up
    t_d = time.perf_counter()
    for t in range(args.desync_steps):
        env.act(actions[(steps_done + t) % T])
        env.observe()
    torch.cuda.synchronize()
    desync_s = time.perf_counter() - t_d
    steps_done += args.desync_steps

    # ---- steady state (the headline)
    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    # the timed region can be as short as 50 ms: give nvidia-smi the very same load first, so that the
    # samples (taken every 25 ms until the timed region ends) describe the clocks it ran at. A fixed
    # number of steps (about a second of the default workload on a B200), not a fixed time, so that
    # the timed steps start from the same env state on every run.
    for _ in range(CLOCK_WARM_ROUNDS):
        for t in range(20):
            env.act(actions[(steps_done + t) % T])
            env.observe()
        torch.cuda.synchronize()
    launches0 = env.kernel_launches()
    elapsed_ms = max_over_ranks(timed_rollout(env, actions, steps_done, K, barrier, gather=args.gather, dist=dist), dist, dev)
    launches = env.kernel_launches() - launches0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(env, args.dump_outputs)
    steps_done += K
    value = n * world * K / (elapsed_ms / 1000.0)
    value_cold = n * world * K / (cold_ms / 1000.0)
    rfrac = reset_fraction(env, actions, steps_done, max(20, min(100, K)))
    steps_done += max(20, min(100, K))
    checksum = int(env.observe()[1]["rgb"].sum().item())
    errors = env.errors()

    # ---- roofline pass: the same steps with every kernel launched back to back on one stream (one
    # launch per game covering all its envs) and CUDA events recorded around each launch on that
    # stream, so a kernel's duration is its own. In the throughput loop above launches of different
    # env chunks overlap on the SMs and an event pair would also count the neighbours' time.
    Kr = max(5, min(20, K))
    env.set_launch_shape(chunks=1, serialize=True)
    for t in range(3):
        env.act(actions[t % T])
        env.observe()
    env.kernel_timing_begin(Kr * 64)
    for t in range(Kr):
        env.act(actions[(W + t) % T])
        env.observe()
    ktimes = env.kernel_timing_end()
    env.set_launch_shape(chunks=0, serialize=False)
    env.close()

    # ---- e2e: the reference-facing C ABI with host buffers, H2D/D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        from procgen_b200.numa import pin_to_gpu_numa_node

        saved_affinity = os.sched_getaffinity(0)
        numa = pin_to_gpu_numa_node(torch.cuda.current_device()) if not args.no_numa_pin else {"pinned": False}
        Ke = max(3, min(args.e2e_steps, K))
        henv = ProcgenGym3Env(n, args.game, distribution_mode=args.mode, num_levels=0, start_level=0, rand_seed=0,
                              shard=(rank, world) if world > 1 else None, host_buffers=True)
        host_actions = actions[: W + Ke].cpu().numpy()
        for t in range(min(W, 3)):
            henv.act(host_actions[t])
            henv.observe()
        barrier()
        t0 = time.perf_counter()
        for t in range(Ke):
            henv.act(host_actions[W + t])
            rew_h, ob_h, first_h = henv.observe()
        barrier()
        el = max_over_ranks(time.perf_counter() - t0, dist, dev)
        d2h = (64 * 64 * 3 + 4 + 1 + 4 + 1 + 4) * n
        e2e = {"value": n * world * Ke / el, "unit": "env-steps/s", "h2d_bytes_per_step": 4 * n * world,
               "d2h_bytes_per_step": d2h * world, "steps": Ke, "d2h_gbs_per_rank": d2h * Ke / el / 1e9,
               "numa": numa, "api": "libenv_act + libenv_observe (host numpy buffers, page-locked)", "timer": "host perf_counter around the calls",
               "note": "cold start (synchronised episodes); PCIe-bound, so level generation does not show"}
        henv.close()
        os.sched_setaffinity(0, saved_affinity)   # the CPU baseline below gets every core back

    # ---- BASELINE configs[4] riding along on multi-GPU runs: the 16-game list, 32 768 envs per GPU,
    # without and with the per-step NCCL gather of every rank's rgb shard to rank 0
    config5 = None
    if args.config5 or (world > 1 and not args.no_config5 and "," not in args.game):
        try:
            n5 = 32768
            env5 = ProcgenGym3Env(n5, ALL16, distribution_mode="hard", num_levels=0, start_level=0, rand_seed=0,
                                  shard=(rank, world) if world > 1 else None)
            act5 = torch.randint(0, 15, (64, n5), device=dev, dtype=torch.int32, generator=gen)
            env5.observe()
            K5 = max(10, min(30, K))
            for t in range(args.config5_desync):
                env5.act(act5[t % 64])
                env5.observe()
            ms_plain = max_over_ranks(timed_rollout(env5, act5, 0, K5, barrier), dist, dev)
            config5 = {"workload": f"16-game list, {n5} envs/GPU x {world} GPUs = {n5 * world} envs, hard, after {args.config5_desync} "
                                   "desync steps", "steps": K5,
                       "value": n5 * world * K5 / (ms_plain / 1000.0), "ms_per_step": ms_plain / K5, "unit": "env-steps/s"}
            if dist is not None:
                if not args.nccl_gather:
                    env5.enable_peer_gather(0)
                for t in range(2):
                    env5.act(act5[t])
                    env5.observe()
                    env5.gather_observations(0)
                ms_g = max_over_ranks(timed_rollout(env5, act5, 0, K5, barrier, gather=True, dist=dist), dist, dev)
                config5["with_gather"] = {"value": n5 * world * K5 / (ms_g / 1000.0), "ms_per_step": ms_g / K5,
                                          "gather_bytes_per_step_into_rank0": (world - 1) * n5 * 64 * 64 * 3,
                                          "how": env5.gather_how()}
            config5["env_error_bits"] = env5.errors()
            env5.close()
        except Exception as e:  # noqa: BLE001 - the secondary record must never take the headline down with it
            config5 = {"error": repr(e)[:300]}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peak, peak_kind = measured_peak_gbs()
    # Dominant kernel = render_kernel (writes the observations). One launch renders `envs_per_launch`
    # frames = 12 288 algorithmic bytes each (SURVEY §8d); its duration comes from the roofline pass.
    pairs = max(1, ktimes["launch_pairs"])
    render_ms_avg = ktimes["render_ms"] / pairs
    logic_ms_avg = ktimes["logic_ms"] / pairs
    setup_ms_avg = ktimes["setup_ms"] / pairs
    envs_per_launch = ktimes["env_steps"] / pairs
    algo_bytes_per_launch = ALGO_BYTES_PER_ENV_STEP * envs_per_launch
    achieved = algo_bytes_per_launch / (render_ms_avg / 1000.0) / 1e9 if render_ms_avg > 0 else 0.0
    step_ms = elapsed_ms / K
    # DRAM bytes of ONE render_kernel launch from an `ncu --set full` capture taken at exactly this
    # launch size (profiles/traffic_r02.json says which command produced it); null for any other shape
    traffic = None
    traffic_src = None
    tpath = os.path.join(ROOT, "profiles", "traffic_r02.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            ent = tj.get(f"{args.game}:{args.mode}:{int(envs_per_launch)}")
            if ent:
                traffic = ent["dram_bytes_per_launch"]
                traffic_src = ent.get("source")
        except Exception:
            traffic = None
    cpu = None
    from oracle.ref_env import REF_LIB

    if not os.path.exists(REF_LIB):
        cpu = {"value": None, "note": "not measured: oracle/_ref (built from the reference tree) is absent"}
    elif not args.no_cpu_baseline:
        rate, detail = cpu_reference_rate(args.game, args.mode, budget_s=args.cpu_budget)
        cpu = {"value": rate, "unit": "env-steps/s", "cores": detail["cores"], "kind": "reference", "host": host_cpu_info(),
               "sample": detail["sample"] + "; reference game logic compiled unmodified + Qt raster restated on CPU"}
    out = {
        "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32+u8", "data": "synthetic", "config": workload_config(args),
        "value_cold": value_cold, "ms_per_step_cold": cold_ms / K,
        "steady_state": {"desync_steps": args.desync_steps, "desync_seconds": desync_s,
                         "episode_end_fraction_per_step": rfrac,
                         "note": "value = after the desync rollout (episode boundaries and level generation spread over "
                                 "steps); value_cold = first K steps after the synchronised initial reset"},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_kind": peak_kind,
                     "kernel": f"render_kernel<{args.game}>",
                     "kernel_ms_avg": render_ms_avg, "launches_timed": ktimes["launch_pairs"], "envs_per_launch": envs_per_launch,
                     "algorithmic_bytes_per_launch": algo_bytes_per_launch,
                     "logic_kernel_ms_avg": logic_ms_avg, "setup_kernel_ms_avg": setup_ms_avg, "step_ms_avg": step_ms,
                     "how": "CUDA events around each launch, launches serialised on one stream (separate pass of %d steps, "
                            "steady state)" % Kr,
                     "whole_step_achieved": ALGO_BYTES_PER_ENV_STEP * n / (step_ms / 1000.0) / 1e9},
        "cpu_baseline": cpu, "obs_checksum": checksum, "env_error_bits": errors,
    }
    if config5 is not None:
        out["config5"] = config5
    print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()


ALL16 = ("bigfish,bossfight,caveflyer,chaser,climber,coinrun,dodgeball,fruitbot,heist,jumper,leaper,maze,"
         "miner,ninja,plunder,starpilot")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--game", default="coinrun")
    ap.add_argument("--mode", default="easy")
    ap.add_argument("--envs-per-gpu", type=int, default=65536)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--cpu-budget", type=float, default=15.0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-numa-pin", action="store_true", help="e2e leg: do not pin the process to the GPU's NUMA node")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--desync-steps", type=int, default=1500,
                    help="untimed rollout before the steady-state measurement (episodes ~500-1000 steps)")
    ap.add_argument("--chunks", type=int, default=0, help="profiling aid: env chunks per step (0 = library default)")
    ap.add_argument("--config5", action="store_true", help="also measure BASELINE configs[4] (16-game list, 32768 envs/GPU)")
    ap.add_argument("--no-config5", action="store_true")
    ap.add_argument("--config5-desync", type=int, default=300)
    ap.add_argument("--nccl-gather", action="store_true", help="keep the plain NCCL gather (no peer writes) for the gather measurements")
    ap.add_argument("--gather", action="store_true",
                    help="BASELINE configs[4] variant: NCCL-gather every step's rgb shard to rank 0 inside the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the observe() outputs of the last steady-state timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.game == "all16":  # BASELINE configs[4]: env n plays game n % 16
        args.game = ALL16
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
