#!/usr/bin/env python
"""Benchmark of the hot path: env-steps/sec of the batched DeepMimic step (BASELINE.json metric).

One "step" = one 30 Hz policy step of every environment on this rank: set_action -> 20 x Update(1/600)
(= 40 dynamics sub-steps) -> record_state + calc_reward + flags -> reset of finished episodes, and for N > 1 one
exchange of [obs | reward | done] rows between the ranks.  value = policy steps of all ranks / max-over-ranks device time.
Both arms run the SURVEY.md 8(d) workload: random-policy actions, 20 s episode limit, falls end episodes and reset the environment.

  python bench.py --gpus 1 --steps 64 --warmup 4            # this framework (CUDA path through the C ABI)
  python bench.py --impl reference --gpus 1 --steps 3       # CPU restatement of the reference path on all usable host cores
  python bench.py --arg-file args/train_dog3d_trot_args.txt # BASELINE.json configs[3] (2048 envs, 64-dof quadruped)
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

ALG_BYTES_PER_UPDATE = {"humanoid3d": 792, "dog3d": 1528}   # SURVEY.md 8(d): fp32 words read+written per Update(1/600) per env
# per policy step on top of the 20 updates: action read + observation write + reward / done (SURVEY.md 8(d))
ALG_IO_BYTES_PER_STEP = {"humanoid3d": 4 * (28 + 227 + 2), "dog3d": 4 * (58 + 347 + 2)}
FP32_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12           # 148 SMs x 128 fp32 lanes x 2 (FMA) x 1.965 GHz: CUDA-core fp32 peak of a B200


def metric_name(char, clip, envs):
    return "env-steps/sec (30 Hz policy steps; %s_%s, %d envs/GPU)" % (char, clip, envs)


def usable_cores():
    """host cores this process may use: the affinity mask capped by the cgroup cpu quota (os.cpu_count() counts the whole box and
    oversubscribed the 1-GPU lease in round 1)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        txt = open("/sys/fs/cgroup/cpu.max").read().split()
        if txt and txt[0] != "max":
            n = min(n, max(1, int(float(txt[0]) / float(txt[1]))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=0, help="default: 4096 (humanoid3d) / 2048 (dog3d), the BASELINE.json configs")
    ap.add_argument("--arg-file", default="args/train_humanoid3d_spinkick_args.txt")
    ap.add_argument("--preroll", type=int, default=48, help="untimed policy steps before the warm-up: the timed region then sees the steady-state mix of "
                    "stance / flight / falling characters, not 4096 freshly reset ones")
    ap.add_argument("--episode-seconds", type=float, default=20.0, help="episode time limit of both arms (SURVEY.md 8d)")
    ap.add_argument("--cpu-baseline-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--updates-per-launch", type=int, default=20)
    ap.add_argument("--exchange", default="auto", choices=["auto", "nccl", "p2p"], help="N > 1: how the [obs | reward | done] rows reach the other ranks")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (observation / reward / done rows, flags, and the goal, AMP "
                         "observation and imitation reward of the AMP scenes) as DIR/<name>.npy; the inputs are seeded, so two builds can be compared")
    return ap.parse_args()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, gathered, local, num_envs):
    """gathered: name -> array [world, N, ...]; local: name -> array [N, ...] (this rank's environments).  Written as float32 .npy files.
    Above DUMP_LIMIT_BYTES in all, a fixed seeded sample of the environments is kept (the same ids in every array, listed in env_ids.npy)."""
    arrays = {k: np.asarray(v, dtype=np.float32) for k, v in list(gathered.items()) + list(local.items())}
    per_env = sum(v.nbytes for v in arrays.values()) / num_envs
    keep = None
    if per_env * num_envs > DUMP_LIMIT_BYTES:
        n = max(1, int((DUMP_LIMIT_BYTES - 8 * num_envs) // per_env))
        keep = np.sort(np.random.default_rng(0).choice(num_envs, size=n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        if keep is not None:
            v = v[:, keep] if k in gathered else v[keep]
        np.save(os.path.join(out_dir, k + ".npy"), v)
    if keep is not None:
        np.save(os.path.join(out_dir, "env_ids.npy"), keep.astype(np.float64))


# ----------------------------------------------------------------------------- CPU arm (oracle = port of the reference path)
def scene_args(arg_file):
    """arg list of a bench workload.  The AMP task scenes name a 56-clip, 48 MB dataset that is not in the committed asset archive: they run on
    the authored 56-entry dataset of the same shape (tests/golden/make_assets.py) -- synthetic data, said so in the JSON line."""
    extra = ["--motion_file", "data/datasets/synthetic_locomotion_56.txt"] if "_amp_" in arg_file else []
    return extra + ["--arg_file", arg_file]


def _oracle_worker(arg_file, root, seconds, seed, max_time, q):
    from tests.oracle_binding import Oracle
    from tests.parity_util import random_policy_action
    o = Oracle(scene_args(arg_file), root)
    amp = "_amp_" in arg_file
    off, scl, lo, hi = o.action_statics()
    rng = np.random.default_rng(seed)
    o.reset(float(rng.uniform(0, o.motion_duration)), 0.0, max_time)
    steps = 0
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        o.set_action(random_policy_action(rng, off, scl, lo, hi))
        for _ in range(20):
            o.update(1.0 / 600.0)
            if o.is_episode_end():
                o.reset(float(rng.uniform(0, o.motion_duration)), 0.0, max_time)
                break
        o.record_state(); o.calc_reward()
        if amp:      # config 5: goal, AMP agent observation and the imitation reward next to the task reward
            o.record_goal(); o.record_amp_obs_agent(); o.calc_reward_imitate()
        steps += 1
    q.put((steps, time.perf_counter() - t0))


def cpu_policy_steps_per_sec(arg_file, root, seconds, procs, max_time):
    ctx = mp.get_context("fork")
    q = ctx.Queue()
    ps = [ctx.Process(target=_oracle_worker, args=(arg_file, root, seconds, 100 + i, max_time, q)) for i in range(procs)]
    for p in ps:
        p.start()
    res = [q.get() for _ in ps]
    for p in ps:
        p.join()
    rates = np.array([s / t for s, t in res])
    return float(rates.sum()), rates


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled DURING the timed region: NVML directly (a query takes microseconds, so even a 30 ms region gets
    many samples), nvidia-smi as the fallback (one query takes tens of milliseconds)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons = index, False, [], set()
        self.max_mhz, self.source = None, "nvidia-smi"
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:   # NVML enumerates physical devices
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if index < len(ids) and ids[index].isdigit():
                    idx = int(ids[index])
            self._h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self._nvml, self.source = pynvml, "nvml"
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n = self._nvml
        self.samples.append(float(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)))
        get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons")
        r = int(get(self._h))
        for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20)):   # nvml.h nvmlClocksEventReason*
            if r & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=5).stdout.strip().split(",")
        self.samples.append(float(out[0])); self.max_mhz = float(out[1])
        for n, v in zip(names, out[2:]):
            if "Active" in v and "Not" not in v:
                self.reasons.add(n)

    def run(self):
        while not self.stop_flag:
            try:
                if self._nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                if self._nvml is not None:      # NVML query failed: fall back to nvidia-smi for the rest of the run
                    self._nvml, self.source = None, "nvidia-smi"
                    continue
            time.sleep(0.002 if self._nvml is not None else 0.2)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples), "source": self.source}


def _profile_facts(char):
    """ncu-derived facts about the dominant kernel (written by tools/ncu_summary.py from the round's `ncu --set full` capture of this same
    command; static between captures -- the file names the capture it came from)"""
    try:
        d = json.load(open(os.path.join(REPO, "profiles", "step_metrics_%s.json" % char)))
        return d
    except Exception:
        return {}


def main():
    a = parse()
    from deepmimic_b200.assets import asset_root
    root = asset_root(prefer_archive=True)   # the committed archive: the same inputs here and on the GPU box
    char = "dog3d" if "dog" in a.arg_file else "humanoid3d"
    amp = "_amp_" in a.arg_file
    base = os.path.basename(a.arg_file)
    clip = base.replace("train_", "").replace("run_", "").replace("_args.txt", "").replace(char + "_", "").replace("amp_", "amp-")
    if a.envs_per_gpu <= 0:
        a.envs_per_gpu = 2048 if char == "dog3d" else 4096
    N = a.envs_per_gpu
    METRIC = metric_name(char, clip, N)
    workload = "%s / %s, %d envs/GPU, random-policy actions, 20 x Update(1/600) per step, %.0f s episode limit, falls reset the environment" % (base, char, N, a.episode_seconds)
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if a.impl == "reference":
        if rank != 0:
            return 0
        cores = usable_cores()
        # each "step" is a bounded sample: all usable host cores run independent single-env episodes for a fixed wall time
        per_step_seconds = max(0.3, min(20.0, 90.0 / max(1, a.steps + a.warmup)))   # whole run ~90 s whatever K and W are
        vals, per_proc = [], []
        for s in range(a.warmup + a.steps):
            v, rates = cpu_policy_steps_per_sec(a.arg_file, root, per_step_seconds, cores, a.episode_seconds)
            if s >= a.warmup:
                vals.append(v); per_proc.append(rates)
        value = float(np.mean(vals))
        pp = np.concatenate(per_proc)
        line = {"metric": METRIC, "value": value, "unit": "policy_steps/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": 1000.0 * per_step_seconds, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64+f32", "data": "synthetic",
                "impl": "reference", "config": {"workload": workload, "note": "CPU restatement of the reference path (oracle port, not Bullet): the reference itself needs Bullet 2.88 + Eigen, absent here",
                                                "host_cpu_count": os.cpu_count(), "usable_cores": cores,
                                                "per_process_policy_steps_per_s": {"min": float(pp.min()), "median": float(np.median(pp)), "max": float(pp.max())}},
                "cpu_baseline": {"value": value, "unit": "policy_steps/s", "cores": cores, "kind": "port",
                                 "sample": "%d processes (affinity / cgroup core count; the box has %d) x %.1f s of single-env episodes per step (process replication = the reference's only parallelism, mpi_run.py)"
                                           % (cores, os.cpu_count() or 0, per_step_seconds)},
                "e2e": {"value": value, "unit": "policy_steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    from deepmimic_b200.capi import BatchedCore
    from deepmimic_b200.sharding import make_exchange
    assert torch.cuda.is_available(), "bench.py --impl b200 needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    core = BatchedCore(scene_args(a.arg_file), N, root, device=local_rank, seed=1000 + rank, global_env_offset=rank * N)
    S, A = core.dims.state_size, core.dims.action_size
    stream = torch.cuda.ExternalStream(core.stream(), device=local_rank)
    dt = 1.0 / 600.0
    upl = a.updates_per_launch
    with torch.cuda.stream(stream):
        # random-policy action bank (zero-mean in the agent's normalised action space, clipped to the bounds)
        g = torch.Generator(device="cuda"); g.manual_seed(7 + rank)
        off = torch.tensor(core.static(2), dtype=torch.float32, device="cuda"); scl = torch.tensor(core.static(3), dtype=torch.float32, device="cuda")
        lo = torch.tensor(core.static(4), dtype=torch.float32, device="cuda"); hi = torch.tensor(core.static(5), dtype=torch.float32, device="cuda")
        bank = 16
        actions = torch.clamp(-off + 0.25 / scl * torch.randn(bank, N, A, device="cuda", generator=g), lo, hi).contiguous()
        flags = torch.zeros(N, 4, dtype=torch.int32, device="cuda")
        if amp:
            goal_buf = torch.zeros(N, max(1, core.dims.goal_size), device="cuda"); amp_buf = torch.zeros(N, core.dims.amp_obs_size, device="cuda"); rim_buf = torch.zeros(N, device="cuda")
        xchg = make_exchange(a.exchange, core, N, S, rank, world, torch.device("cuda", local_rank))   # owns the [obs | reward | done] rows of every rank
        flush = torch.empty(192 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")   # > 126 MB L2
        flag_sums = torch.zeros(N, 4, dtype=torch.int32, device="cuda")
        # episodes: fixed 20 s limit in both arms (the train args anneal 0.5 s -> 20 s over 32 M samples; the end of the schedule is the workload)
        big = np.full(N, a.episode_seconds)
        core.reset(True, max_time=big)
        core.set_episode_limit(a.episode_seconds)

        def step(i, ev=None):
            core.set_action(actions[i % bank])
            if ev: ev[0].record(stream)
            for _ in range(20 // upl):
                core.update(dt, upl)
            if ev: ev[1].record(stream)
            xchg.publish(i)               # record_state + calc_reward + done; N > 1: the rows reach all ranks (P2P stores over NVLink, or one NCCL all-gather)
            core.flags(flags)
            if amp:                       # config 5: goal + AMP agent observation + imitation reward (active clip) recorded alongside
                core.record_goal(goal_buf); core.amp_obs_agent(amp_buf); core.reward_imitate(rim_buf)
            flag_sums.add_(flags)         # per-environment counts of done / terminate flags (one small kernel; summed after the timed region)
            if i > 0:
                xchg.consume(i - 1)       # the learner's side of the exchange: all ranks' rows of the previous step have arrived, slot released
            core.reset(False)

        for i in range(a.preroll + a.warmup):
            step(i)
        stream.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        flag_sums.zero_()
        sampler = ClockSampler(local_rank); sampler.start()
        l0 = core.counters()[0]
        step_ms, upd_ms = [], []
        for i in range(a.steps):
            flush.fill_(float(i))            # L2 flush between timed iterations (outside the event pairs)
            e0, e1, ek0, ek1 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
            e0.record(stream)
            step(a.preroll + a.warmup + i, (ek0, ek1))
            e1.record(stream)
            step_ms.append((e0, e1)); upd_ms.append((ek0, ek1))
        xchg.consume(a.preroll + a.warmup + a.steps - 1)
        stream.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        sampler.stop_flag = True; sampler.join(timeout=2)
        launches = core.counters()[0] - l0 + a.steps * xchg.launches_per_step
        if a.dump_outputs and rank == 0:
            obs, rew, done = xchg.rows(a.preroll + a.warmup + a.steps - 1)
            local = {"flags": flags}
            if amp:
                local.update(amp_obs_agent=amp_buf, reward_imitate=rim_buf)
                if core.dims.goal_size:
                    local["goal"] = goal_buf
            stream.synchronize()
            dump_outputs(a.dump_outputs, {k: v.cpu().numpy() for k, v in (("obs", obs), ("reward", rew), ("done", done))},
                         {k: v.cpu().numpy() for k, v in local.items()}, N)
        per_step = np.array([x.elapsed_time(y) for x, y in step_ms])
        per_kern = np.array([x.elapsed_time(y) for x, y in upd_ms]) / (20 // upl)
        total_ms = float(per_step.sum())
        kern_ms = float(per_kern.mean())
        t = torch.tensor([total_ms, -kern_ms, kern_ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t[0].item()); kern_min_rank, kern_max_rank = -float(t[1].item()), float(t[2].item())
        overflow = core.counters()[1]
        done_count, fell_count = int(flag_sums[:, 1].sum().item()), int((flag_sums[:, 2] > 0).sum().item()) if amp else int(flag_sums[:, 2].sum().item())

        # ---- end-to-end through the host-buffer C-ABI call (page-locked caller buffers, H2D actions + D2H obs/reward/flags every step)
        nb = 4
        t_acts = [actions[k].cpu().pin_memory() for k in range(nb)]
        t_obs = torch.zeros(N, S, dtype=torch.float32).pin_memory()
        t_rew = torch.zeros(N, dtype=torch.float32).pin_memory(); t_fl = torch.zeros(N, 4, dtype=torch.int32).pin_memory()
        h_acts, h_obs, h_rew, h_fl = [x.numpy() for x in t_acts], t_obs.numpy(), t_rew.numpy(), t_fl.numpy()
        for k in range(3):
            core.step_host(h_acts[k % nb], dt, 20, h_obs, h_rew, h_fl, reset_done=True)
        core.sync()
        ke = max(64, a.steps // 2)     # at least 64 calls (~0.13 s): the wall-clock figure must not be dominated by start-up skew between ranks
        if world > 1:
            torch.cuda.synchronize()
            dist.barrier()             # NCCL's barrier is stream-ordered: synchronise again so that it has completed before the clock starts
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(ke):
            core.step_host(h_acts[i % nb], dt, 20, h_obs, h_rew, h_fl, reset_done=True)
        core.sync()
        e2e_s = time.perf_counter() - t0
        te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_value = world * N * ke / float(te.item())
        # phase breakdown of the same call (separate short pass with the library's event hooks on; not part of the timed e2e figure)
        core.set_timing(True)
        br = []
        for i in range(8):
            core.step_host(h_acts[i % nb], dt, 20, h_obs, h_rew, h_fl, reset_done=True)
            br.append(core.step_host_timing())
        core.set_timing(False)
        e2e_break = {k: float(np.median([b[k] for b in br])) for k in br[0]}

    value = world * N * a.steps / (total_ms / 1000.0)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs", 6650.0)
    io_bytes = ALG_IO_BYTES_PER_STEP[char] + (4 * (core.dims.amp_obs_size + core.dims.goal_size + 1) if amp else 0)
    alg_bytes = N * (upl * ALG_BYTES_PER_UPDATE[char] + io_bytes * upl // 20)
    achieved = alg_bytes / (kern_ms / 1000.0) / 1e9
    pf = _profile_facts(char)
    flop_per_update = pf.get("fp32_flop_per_update_per_env")
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": pf.get("dram_bytes_per_launch"),
            "kernel": "dm_step_kernel", "kernel_ms": kern_ms, "algorithmic_bytes_per_launch": alg_bytes,
            "algorithmic_bytes_note": "%d envs x (%d updates x %d B + %d B action/obs/reward I/O of the policy step)" % (N, upl, ALG_BYTES_PER_UPDATE[char], io_bytes * upl // 20),
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
            "note": "latency/issue-bound path: state stays on chip for the whole launch, HBM fraction is small by construction (SURVEY 8d); the issue / fp32 figures below are the informative ones",
            "issue_slot_pct_of_peak": pf.get("issue_slot_pct_of_peak"), "sm_active_pct": pf.get("sm_active_pct"),
            "profile_source": pf.get("source")}
    if flop_per_update:
        tf = flop_per_update * N * upl / (kern_ms / 1000.0) / 1e12
        roof.update({"fp32_flop_per_update_per_env": flop_per_update, "fp32_tflops": tf, "fp32_peak_tflops": FP32_PEAK_TFLOPS, "fp32_frac": tf / FP32_PEAK_TFLOPS,
                     "fp32_flop_source": pf.get("flop_source")})
    line = {"metric": METRIC, "value": value, "unit": "policy_steps/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": total_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic" + (" (56-entry clip dataset of the reference's shape over the archive's locomotion clips)" if amp else ""),
            "config": {"workload": workload, "sim_updates_per_s": value * 20, "l2": "flushed between timed steps (192 MiB fill)", "updates_per_launch": upl,
                       "preroll_steps": a.preroll, "episode_limit_s": a.episode_seconds,
                       "episodes_finished_in_timed_region": done_count, "of_which_falls": fell_count, "solver_row_overflows": overflow,
                       "step_ms": {"min": float(per_step.min()), "median": float(np.median(per_step)), "max": float(per_step.max())},
                       "kernel_ms_over_ranks": {"min": kern_min_rank, "max": kern_max_rank},
                       "e2e_host_buffers": "page-locked caller buffers, DMA'd directly by dm_step_host (pageable ones would pass through pinned staging); %d action buffers in rotation; finished episodes reset inside the call" % nb,
                       "e2e_breakdown_ms": e2e_break,
                       "collective": xchg.describe() if world > 1 else "none (1 GPU)"},
            "roofline": roof,
            "e2e": {"value": e2e_value, "unit": "policy_steps/s", "h2d_bytes_per_step": int(N * A * 4), "d2h_bytes_per_step": int(N * (S + 1 + 4) * 4)},
            "gpu_launches": int(launches), "clocks": sampler.summary()}
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        v, _ = cpu_policy_steps_per_sec(a.arg_file, root, a.cpu_baseline_seconds, 1, a.episode_seconds)
        line["cpu_baseline"] = {"value": v, "unit": "policy_steps/s", "cores": 1, "kind": "port",
                                "sample": "1 process x %.0f s of single-env episodes with the same action distribution and episode limit (CPU restatement, not Bullet)" % a.cpu_baseline_seconds}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        xchg.close()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
