#!/usr/bin/env python
"""bench.py — env-steps/s of the batched QuadX-Hover stepper (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            (ours; torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  (CPU arm: the oracle port, all host threads)
    python bench.py ... --dump-outputs DIR                   (also write what the last timed step returned, DIR/<name>.npy)

One "step" = one env.step() of every env of this rank's shard = ONE k_hover_step launch (6 physics substeps,
3 control ticks, reward / termination / observation fused; finished envs are reset by their own thread on the next
call, and builder CTAs appended to the same grid rebuild the spare post-reset states that were consumed).
Workload (config.workload): QuadX-Hover-v4, mode 0, 65 536 envs per GPU, uniform random actions in the env's action
box, NEXT_STEP autoreset — BASELINE.json configs[1].  Prints ONE JSON line on rank 0.  R blocks of exactly K steps
are timed (L2 flushed between steps, per-step CUDA-event pairs); `value` is the median block.  Under torchrun the line
also carries config.value_strong_65536_total (BASELINE's 65 536 envs in total, split over the ranks) and
config.dogfight_split (configs[4] with an arena's aircraft on different ranks: exchange every Aviary step).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.realpath(__file__))
sys.path.insert(0, ROOT)

ALGO_BYTES_PER_ENV_STEP = 330  # SURVEY.md §8(d): 2*4*28 state + 16 action + 84 obs + 6 reward/flags
ENVS_PER_GPU = 65536


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def _ncu_summary_path():
    """newest committed `ncu --set full` summary of the step kernel (profiles/rNN_k_hover_step_ncu_summary.txt), or None"""
    import glob

    found = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_k_hover_step_ncu_summary.txt")))
    return found[-1] if found else None


def ncu_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture (profiles/), or None."""
    path = _ncu_summary_path()
    try:
        total, seen = 0.0, 0
        for line in open(path):
            f = line.split()
            if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[f[2]]
                total += float(f[1]) * mult
                seen += 1
                if seen == 2:  # the first kernel block of the summary is the step launch
                    return total
    except Exception:
        pass
    return None


def ncu_flops():
    """(fp32, fp64) FLOPs per step launch from the committed ncu capture, or (None, None)."""
    path = _ncu_summary_path()
    out = {}
    try:
        for line in open(path):
            f = line.split()
            if len(f) >= 3 and f[0] == "derived:" and f[1] not in out:
                out[f[1]] = float(f[2])
    except Exception:
        pass
    return out.get("fp32_flops_per_launch"), out.get("fp64_flops_per_launch")


def ncu_warp_instructions():
    """warp instructions of one step launch (smsp__inst_executed.sum of the committed ncu capture), or None"""
    try:
        for line in open(_ncu_summary_path()):
            f = line.split()
            if len(f) >= 2 and f[0] == "smsp__inst_executed.sum":
                return float(f[1])
    except Exception:
        pass
    return None


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def host_threads() -> int:
    """Threads this process may actually use: affinity mask and cgroup CPU quota, not just the core count."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    try:  # cgroup v2, then v1
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0:
                n = max(1, min(n, quota // period))
        except Exception:
            pass
    return n


def tune_oracle_threads(o, L) -> int:
    """The CPU arm gets its best thread count: short probes at 1x, 1/2x, 1/4x, 1/8x of the usable threads (SMT siblings and
    memory bandwidth make 'all of them' the wrong answer on some hosts)."""
    n = host_threads()
    best, best_rate = n, 0.0
    for t in sorted({n, max(1, n // 2), max(1, n // 4), max(1, n // 8)}, reverse=True):
        L.orc_set_num_threads(t)
        o.env_rollout(2)
        t0 = time.perf_counter()
        done = o.env_rollout(6)
        rate = done / (time.perf_counter() - t0)
        if rate > best_rate:
            best, best_rate = t, rate
    L.orc_set_num_threads(best)
    return best


def cpu_oracle_rate(envs: int, target_seconds: float, threads: int | None = None):
    """env-steps/s of the CPU oracle port on the host cores; bounded sample of the same workload."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np

    from engines import build_model, hover_config
    from oracle import oracle as orc_mod

    L = orc_mod.lib()
    L.orc_set_num_threads(int(threads) if threads else host_threads())
    model = build_model("quadx", "cf2x")
    env = hover_config(0, "quaternion", False, 3.0, autoreset=True)
    o = orc_mod.Oracle(model, env, n=envs, seed=1, start_pos=np.array([0.0, 0.0, 1.0]), start_orn=np.zeros(3))
    o.env_reset()
    if not threads:
        tune_oracle_threads(o, L)
    cores = int(L.orc_num_threads())
    o.env_rollout(5)  # warm-up
    steps, done, chunk = 0, 0, 20
    t0 = time.perf_counter()
    while True:
        done += o.env_rollout(chunk)
        steps += chunk
        dt = time.perf_counter() - t0
        if dt >= target_seconds:
            break
    return done / dt, cores, steps, dt


WORKLOAD = ("QuadX-Hover-v4 (BASELINE configs[1]): flight mode 0, 65536 envs per GPU and step, uniform random actions, NEXT_STEP autoreset, "
            "6 physics substeps + 3 control ticks per env-step")


def base_config(world: int, n: int) -> dict:
    """keys shared by both arms (the driver compares them)"""
    return {"workload": WORKLOAD, "envs_per_gpu": n, "global_envs": world * n, "parallelism": f"env-shard x{world} (no data-path collective)"}


def run_reference(args, rank, world):
    """CPU arm: the reference's algorithm (oracle port; PyBullet itself is not installable here) timed
    on the box's host cores, same metric and config (the same GLOBAL number of envs as our arm steps); rank 0 only."""
    if rank != 0:
        return
    envs = args.envs * world
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np

    from engines import build_model, hover_config
    from oracle import oracle as orc_mod

    L = orc_mod.lib()
    L.orc_set_num_threads(host_threads())  # torchrun exports OMP_NUM_THREADS=1: use the host's threads anyway
    model = build_model("quadx", "cf2x")
    env = hover_config(0, "quaternion", False, 3.0, autoreset=True)
    o = orc_mod.Oracle(model, env, n=envs, seed=1, start_pos=np.array([0.0, 0.0, 1.0]), start_orn=np.zeros(3))
    o.env_reset()
    tune_oracle_threads(o, L)
    cores = int(L.orc_num_threads())
    for _ in range(args.warmup):
        o.env_rollout(1)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        o.env_rollout(1)
    dt = time.perf_counter() - t0
    value = envs * args.steps / dt
    line = {
        "impl": "reference", "metric": "env-steps/s", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": base_config(world, args.envs),
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} steps x {envs} envs of the full workload (oracle/pfb_oracle.c, fp64, OpenMP; thread count tuned by a short probe)"},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def _median(x):
    x = sorted(x)
    return x[len(x) // 2]


def dogfight_split_block(rank, world, dev, steps=40, arenas=8192):
    """BASELINE configs[4] as written: 8192 arenas x 2 agents with an arena's two aircraft on DIFFERENT ranks, one exchange per
    Aviary step (4 per env step).  Times every exchange flavour and checks bit-equality with a single-rank run."""
    import torch
    import torch.distributed as dist

    from pyflyt_b200.pz_envs import MAFixedwingDogfightSplitEnv

    out = {"arenas": arenas, "agents": 2 * arenas, "ranks": world, "collectives_per_step": 4, "payload_bytes_per_agent_per_exchange": 80}
    # ---- parity: every rank steps its slice (Philox noise keyed by global agent id), rank 0 repeats all of it alone
    pa, ps = 1024, 6
    g = torch.Generator().manual_seed(7)
    acts = (torch.rand((ps, 2 * pa, 4), generator=g) * 2 - 1) * 0.4
    kw = dict(seed=3, lethal_distance=150.0, lethal_angle_radians=1.0, damage_per_hit=0.05)

    def run(env):
        lo, hi = env.first_gid, env.first_gid + env.n_local
        obs = [env.reset().clone()]
        rew = []
        for k in range(ps):
            o, r, _, _ = env.step(acts[k, lo:hi].to(dev))
            obs.append(o.clone())
            rew.append(r.clone())
        env.close()
        return torch.stack(obs), torch.stack(rew)

    ok = True
    for ex in ("nccl", "peer-signal"):
        o, r = run(MAFixedwingDogfightSplitEnv(pa, device=dev, exchange=ex, **kw))
        parts_o = [torch.empty_like(o) for _ in range(world)]
        parts_r = [torch.empty_like(r) for _ in range(world)]
        dist.all_gather(parts_o, o.contiguous())
        dist.all_gather(parts_r, r.contiguous())
        if rank == 0:
            so, sr = run(MAFixedwingDogfightSplitEnv(pa, device=dev, single_rank=True, exchange="nccl", **kw))
            ok = ok and bool(torch.equal(torch.cat(parts_o, dim=1), so)) and bool(torch.equal(torch.cat(parts_r, dim=1), sr))
        dist.barrier()
    out["parity_ok"] = ok
    # ---- timing (L2 flushed between steps, per-step event pairs, max over ranks)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    for ex in ("nccl", "peer", "peer-signal"):
        env = MAFixedwingDogfightSplitEnv(arenas, seed=1, device=dev, exchange=ex)
        env.reset()
        act = torch.rand(env.n_local, 4, device=dev) * 2 - 1
        for _ in range(5):
            env.step(act)
        torch.cuda.synchronize(dev)
        dist.barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for k in range(steps):
            flush.fill_(float(k))
            ev[k][0].record()
            env.step(act)
            ev[k][1].record()
        torch.cuda.synchronize(dev)
        t = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        us = float(t[0]) * 1e3 / steps
        out[ex] = {"us_per_step": us, "agent_steps_per_s": 2 * arenas / (us * 1e-6)}
        env.close()
        dist.barrier()
    best = min(("nccl", "peer", "peer-signal"), key=lambda e: out[e]["us_per_step"])
    out.update({"exchange": best, "us_per_step": out[best]["us_per_step"], "agent_steps_per_s": out[best]["agent_steps_per_s"], "steps": steps})
    return out


DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def timed_step_outputs(env) -> dict:
    """What env.step() returned for the batch of the last timed step, as float32 host arrays.  Above DUMP_LIMIT_BYTES only a
    fixed, seeded sample of the envs is kept; `env_index` (float64) says which."""
    import numpy as np

    av = env.aviary
    bits = av.info_bits.cpu().numpy()
    out = {
        "obs": av.obs.cpu().numpy(), "reward": av.reward.cpu().numpy(),
        "terminated": av.term.cpu().numpy().astype(np.float32), "truncated": av.trunc.cpu().numpy().astype(np.float32),
        "info_out_of_bounds": (bits & 1).astype(np.float32), "info_collision": ((bits >> 1) & 1).astype(np.float32),
        "info_env_complete": ((bits >> 2) & 1).astype(np.float32),
    }
    n = av.num_drones
    row_bytes = sum(a[0].nbytes for a in out.values()) + 8
    if n * row_bytes > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT_BYTES // row_bytes, replace=False))
        out = {k: v[keep] for k, v in out.items()}
        out["env_index"] = keep.astype(np.float64)
    return out


def write_outputs(directory: str, arrays: dict) -> None:
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    from pyflyt_b200.gym_envs.quadx_hover_env import QuadXHoverVecEnv

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from pyflyt_b200.sharding import shard_range

    n = args.envs
    first, last = shard_range(world * n, rank, world)  # contiguous global env ids per rank; Philox is keyed by them
    assert last - first == n
    env = QuadXHoverVecEnv(num_envs=n, seed=args.seed, device=dev, env_offset=first)
    av = env.aviary
    env.reset()
    K, W, R = args.steps, args.warmup, args.repeats
    # action pool resident in HBM before the timed region (uniform in the action box, quadx_base_env.py:79-102)
    pool = 32
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    lo = torch.tensor([-3.14159265, -3.14159265, -3.14159265, 0.0], device=dev)
    hi = torch.tensor([3.14159265, 3.14159265, 3.14159265, 0.8], device=dev)
    actions = lo + (hi - lo) * torch.rand((pool, n, 4), device=dev, generator=g)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def flushed_block(aviary, steps, acts, off=0):
        """`steps` env steps, L2 flushed before each (outside the event pair), one CUDA-event pair per step; returns ms summed"""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for k in range(steps):
            flush.fill_(float(k))
            ev[k][0].record()
            aviary.env_step(actions=acts[(off + k) % pool])
            ev[k][1].record()
        barrier()
        return float(sum(a.elapsed_time(b) for a, b in ev))

    for k in range(max(W, 30)):  # past the first terminations: resets and spare rebuilds are inside every timed step
        av.env_step(actions=actions[k % pool])
    barrier()

    # ---- timed region A: device-resident inputs LARGER THAN THE L2.  M independent batches of n envs (own state, spares, outputs;
    #      global env ids continue after this rank's first batch) are stepped round-robin, back to back, one launch = one env
    #      step of one batch.  A batch is touched again only after the other M - 1 batches moved ~23 MB each (state tile in / out,
    #      observations, actions, rewards / flags), i.e. (M - 1) x 23 MB > 126 MB: every launch reads its inputs from DRAM.  No
    #      flush kernel and no per-step events inside the region: exactly K steps between ONE event pair, barrier +
    #      synchronize on both sides; R blocks, the MEDIAN block is reported.
    M = max(1, args.batches)
    rot = [env] + [QuadXHoverVecEnv(num_envs=n, seed=args.seed, device=dev, env_offset=(world * j + rank) * n) for j in range(1, M)]
    for e in rot[1:]:
        e.reset()
    for k in range(max(W, 30) * M):  # every batch past its first terminations
        rot[k % M].aviary.env_step(actions=actions[k % pool])
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)

    def rotating_block(steps, off):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for k in range(steps):
            rot[k % M].aviary.env_step(actions=actions[(off + k) % pool])
        e1.record()
        barrier()
        return float(e0.elapsed_time(e1))

    launches0 = sum(e.aviary.launch_count for e in rot)
    block_ms = [rotating_block(K, W + r * K) for r in range(R)]
    launches = (sum(e.aviary.launch_count for e in rot) - launches0) // R
    # the later regions step these batches again: keep what the last timed step returned
    dumped = timed_step_outputs(rot[(K - 1) % M]) if args.dump_outputs and rank == 0 else None
    # ---- region R (context): the same K env steps of the same batches as FUSED rollouts — pfb_env_rollout(16): 16 env steps per
    #      launch with the state in registers, actions drawn on device, every step's observations / rewards / flags written, spares
    #      topped up behind every launch (all inside the event pair); "synthetic random-action rollouts" in BASELINE.json's words
    FUSED_T = 16

    def fused_block(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for c in range(steps // FUSED_T):
            rot[c % M].rollout(FUSED_T)
        e1.record()
        barrier()
        return float(e0.elapsed_time(e1))

    Kf = max(FUSED_T, (K // FUSED_T) * FUSED_T)
    for c in range(2 * M):  # spares three ahead, past the first fused launches
        rot[c % M].rollout(FUSED_T)
    fl0 = sum(e.aviary.launch_count for e in rot)
    fused_ms = _median([fused_block(Kf) for _ in range(min(R, 3))])
    fused_launches = (sum(e.aviary.launch_count for e in rot) - fl0) // min(R, 3)
    for e in rot[1:]:
        e.close()
    # ---- region F (context, round-1 / round-2a protocol): ONE batch, L2 flushed by a 256 MiB write before every step, a CUDA-event
    #      pair per step (each pair carries ~3 us of launch / completion latency that back-to-back launches overlap)
    flushed_ms = _median([flushed_block(av, K, actions, off=W + r * K) for r in range(min(R, 3))])

    # ---- region K: the same flushed steps with the library's event pair tightly around the step launch (roofline leg)
    av.profile_begin(K)
    flushed_block(av, K, actions)
    kern_ms = av.profile_read(K)
    av.profile_begin(0)

    # ---- region A2 (context): back-to-back, L2-warm, one event pair around K steps
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(K):
        av.env_step(actions=actions[k % pool])
    e1.record()
    barrier()
    warm_ms = e0.elapsed_time(e1)

    # ---- region B: end to end through the host-buffer entry of the C-ABI (pinned host memory)
    act_h = [actions[k].cpu().pin_memory() for k in range(4)]
    # one pinned slab, obs | reward | term | trunc back to back like the device side: the library returns it in one D2H copy
    slab_h = torch.empty(av.out_slab_bytes(n, env.obs_dim), dtype=torch.uint8).pin_memory()
    obs_h, rew_h, te_h, tr_h = av.slab_views(slab_h, n, env.obs_dim)
    for k in range(3):
        av.env_step_host(act_h[k % 4], obs_h, rew_h, te_h, tr_h)
    barrier()
    t0 = time.perf_counter()
    for k in range(K):
        av.env_step_host(act_h[k % 4], obs_h, rew_h, te_h, tr_h)
        torch.cuda.synchronize(dev)  # the caller reads obs/reward here
    e2e_copy_s = time.perf_counter() - t0
    barrier()
    # same call, zero-copy flavour: the kernel itself reads the pinned actions and writes the pinned result slab over PCIe
    for k in range(3):
        av.env_step_mapped(act_h[k % 4], obs_h, rew_h, te_h, tr_h)
    barrier()
    t0 = time.perf_counter()
    for k in range(K):
        av.env_step_mapped(act_h[k % 4], obs_h, rew_h, te_h, tr_h)
        torch.cuda.synchronize(dev)
    e2e_mapped_s = time.perf_counter() - t0
    barrier()
    e2e_s = min(e2e_copy_s, e2e_mapped_s)
    clocks = sampler.stop()
    env.close()

    # ---- region S (context, world > 1): STRONG scaling — BASELINE's 65 536 envs in total, split over the ranks
    strong_ms = 0.0
    if world > 1:
        s0, s1 = shard_range(ENVS_PER_GPU, rank, world)
        ns = s1 - s0
        env_s = QuadXHoverVecEnv(num_envs=ns, seed=args.seed, device=dev, env_offset=s0)
        env_s.reset()
        acts_s = actions[:, :ns].contiguous()
        for k in range(30):
            env_s.aviary.env_step(actions=acts_s[k % pool])
        barrier()
        strong_ms = _median([flushed_block(env_s.aviary, K, acts_s) for _ in range(3)])
        env_s.close()

    # ---- reduce: max over ranks
    t = torch.tensor(block_ms + [warm_ms, e2e_s * 1e3, float(sum(kern_ms)), strong_ms, e2e_copy_s * 1e3, e2e_mapped_s * 1e3, flushed_ms, fused_ms], dtype=torch.float64,
                     device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    vals = [float(x) for x in t.tolist()]
    block_ms, (warm_ms, e2e_ms, kern_total_ms, strong_ms, e2e_copy_ms, e2e_mapped_ms, flushed_ms, fused_ms) = vals[:R], vals[R:]
    import threading

    emitted = threading.Lock()

    def emit(split):
        """rank 0 prints THE json line exactly once (also reachable from the watchdog of the split-dogfight block)"""
        if rank != 0 or not emitted.acquire(blocking=False):
            return
        peak, peak_src = load_peaks()
        total_ms = _median(block_ms)
        value = world * n * K / (total_ms * 1e-3)
        # average duration of a step launch over the timed region: the region is K back-to-back launches of the one kernel, so
        # block time / K bounds it from above (it still contains the ~1 us gaps between consecutive launches)
        kern_avg_s = total_ms * 1e-3 / K
        kern_pair_s = kern_total_ms * 1e-3 / max(len(kern_ms), 1)
        achieved = ALGO_BYTES_PER_ENV_STEP * n / kern_avg_s / 1e9
        cfg = base_config(world, n)
        cfg.update({
            "l2": f"inputs larger than the L2: {M} independent batches of {n} envs stepped round-robin, ~23 MB touched per step, {(M - 1) * 23} MB between two "
                  "steps of the same batch vs 126 MB of L2; K back-to-back launches inside ONE event pair (no flush kernel, no per-step events)",
            "batches": M,
            "rollout_fused": {
                "env_steps_per_s": world * n * Kf / (fused_ms * 1e-3), "us_per_step": fused_ms * 1e3 / Kf, "steps_per_launch": FUSED_T, "steps": Kf,
                "launches_per_block": fused_launches, "frac_hbm_roofline": ALGO_BYTES_PER_ENV_STEP * n * Kf / (fused_ms * 1e-3) / 1e9 / peak,
                "note": "pfb_env_rollout(16) on the same rotating batches: k_hover_rollout keeps the state in registers for 16 env steps (one tile load, one "
                        "tile store), draws the actions on device, writes every step's observations / rewards / flags, and k_hover_spare_topup rebuilds the "
                        "spares the launch consumed; pinned to the oracle by tests/test_timed_path_parity.py::test_hover_fused_rollout_matches_oracle and to the "
                        "one-launch-per-step path by tests/test_gpu_parity.py::test_fused_rollout_equals_stepwise.  `value` stays the one-launch-per-step number",
            },
            "value_l2_flushed_event_pairs": world * n * K / (flushed_ms * 1e-3), "ms_per_step_l2_flushed_event_pairs": flushed_ms / K,
            "l2_flushed_note": "the protocol of the earlier rounds (one batch, 256 MiB write before every step, one CUDA-event pair per step, pairs summed): "
                               "each pair carries ~3 us of launch / completion latency that back-to-back launches overlap (profiles/r02_rotation_sweep.jsonl)",
            "repeats": R, "block_ms": block_ms, "statistic": "median block",
            "precision": "fp32 forces/control/obs; quaternion, position, velocity carried as fp64 (hi+lo fp32 words in HBM)",
            "value_l2_warm": world * n * K / (warm_ms * 1e-3), "ms_per_step_l2_warm": warm_ms / K,
            "value_inline_resets": value, "ms_per_step_inline_resets": total_ms / K,
            "reset_pipeline": "ONE launch per env step: finished envs take their spare post-reset state in the launch after they finish, and the spares consumed are rebuilt in two halves by builder CTAs appended to the grids of that launch and the next. All of it is inside the event pairs (value_inline_resets == value; no side stream, no second launch)",
        })
        if world > 1:
            cfg["value_strong_65536_total"] = ENVS_PER_GPU * K / (strong_ms * 1e-3)
            cfg["ms_per_step_strong"] = strong_ms / K
            cfg["strong_note"] = f"BASELINE's 65536 envs in total = {ENVS_PER_GPU // world} per GPU: the launch is latency-bound (one tile per SM or less), so strong scaling is flat"
        if split is not None:
            cfg["dogfight_split"] = split
        line = {
            "metric": "env-steps/s", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": cfg,
            "e2e": {
                "value": world * n * K / (e2e_ms * 1e-3), "unit": "env-steps/s",
                "h2d_bytes_per_step": n * 4 * 4, "d2h_bytes_per_step": n * (env.obs_dim * 4 + 4 + 1 + 1),
                "method": "pfb_env_step_mapped (kernel reads / writes the pinned host buffers, PCIe overlapped with the launch)" if e2e_mapped_ms <= e2e_copy_ms
                else "pfb_env_step_host (H2D copy, launch, one D2H copy of the result slab)",
                "value_copy": world * n * K / (e2e_copy_ms * 1e-3), "value_mapped": world * n * K / (e2e_mapped_ms * 1e-3),
            },
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {
                "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic(),
                "kernel": "k_hover_step<0,false,false,true,false>", "algorithmic_bytes_per_env_step": ALGO_BYTES_PER_ENV_STEP,
                "kernel_avg_us": kern_avg_s * 1e6, "kernel_event_pair_us_l2_flushed": kern_pair_s * 1e6, "peak_source": peak_src,
                "note": "issue/latency-bound kernel: the HBM fraction is reported because BASELINE.json asks for it; see DESIGN.md",
                "traffic_source": f"dram__bytes_read.sum + dram__bytes_write.sum of the step launch in {os.path.relpath(_ncu_summary_path() or 'profiles/', ROOT)} (one ncu --set full capture, cold caches: the state written by the launch is still L2-resident when it ends, so traffic < algorithmic bytes)",
            },
        }
        f32, f64 = ncu_flops()
        if f32:
            # SURVEY 8(d) asks for both fractions: the non-tensor fp32 pipe next to HBM (148 SMs x 128 lanes x 2 x 1.965 GHz)
            peak32 = 148 * 128 * 2 * 1.965e9 / 1e12
            line["roofline"]["fp32"] = {
                "flops_per_launch": f32, "fp64_flops_per_launch": f64, "achieved_tflops": f32 / kern_avg_s / 1e12, "peak_tflops": peak32,
                "frac": f32 / kern_avg_s / 1e12 / peak32,
                "source": "FFMA/FMUL/FADD thread-instruction counters of the step launch in the same ncu capture",
            }
        winst = ncu_warp_instructions()
        if winst:
            # what actually bounds the kernel (DESIGN.md 6): the warp schedulers.  148 SMs x 4 schedulers issue at most one warp
            # instruction per cycle each; frac = the share of those issue slots the launch uses over its measured duration
            slots = 148 * 4 * 1.965e9 * kern_avg_s
            line["roofline"]["issue"] = {
                "warp_instructions_per_launch": winst, "issue_slots_per_launch": slots, "frac": winst / slots,
                "note": "context: smsp__inst_executed.sum of the same ncu capture / (592 schedulers x 1.965 GHz x the measured launch duration)",
            }
        if world == 1 and not args.no_cpu_baseline:
            rate, cores, steps, dt = cpu_oracle_rate(16384, args.cpu_seconds)
            line["cpu_baseline"] = {
                "value": rate, "unit": "env-steps/s", "cores": cores, "kind": "port",
                "sample": f"{steps} env-steps x 16384 envs ({dt:.1f} s) of the same workload on oracle/pfb_oracle.c (fp64, OpenMP; thread count tuned by a short probe)",
            }
        print(json.dumps(line), flush=True)

    # ---- configs[4] (context, world > 1): the split dogfight needs every rank alive at four exchanges per env step.  It runs LAST and
    #      under a watchdog: whatever happens to it (an exception on one rank, a peer that never arrives), the line above is printed
    split = None
    if world > 1 and not args.no_dogfight_split:
        def expired():
            emit({"error": f"split-dogfight block did not finish within {args.split_timeout:.0f} s; skipped"})
            os._exit(0)

        dog = threading.Timer(args.split_timeout, expired)
        dog.daemon = True
        dog.start()
        try:
            split = dogfight_split_block(rank, world, dev)
        except Exception as e:  # noqa: BLE001 - reported in the line, the hover numbers stand
            emit({"error": repr(e)[:300]})
            os._exit(0)
        dog.cancel()
    emit(split)
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU, help="envs per GPU")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--repeats", type=int, default=5, help="blocks of --steps timed steps; the median block is reported")
    ap.add_argument("--no-dogfight-split", action="store_true", help="skip the configs[4] split-dogfight block under torchrun")
    ap.add_argument("--split-timeout", type=float, default=240.0, help="watchdog of the split-dogfight block (s)")
    ap.add_argument("--batches", type=int, default=12,
                    help="independent 65 536-env batches stepped round-robin in the timed region (their working set exceeds the L2: every "
                         "launch finds its inputs in DRAM); 1 = one batch, L2-warm")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (obs, reward, terminated, truncated, info flags; rank 0's "
                         "shard under torchrun) as DIR/<name>.npy in float32; inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
