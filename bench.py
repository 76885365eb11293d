#!/usr/bin/env python
"""Headline benchmark: agent-steps/s of the fused env-step kernel (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

N=1 runs in-process; for N>1 launch with torch.distributed.run (one rank per GPU, NCCL only for
the barrier / max-over-ranks reduction -- the env path has no data-path collective: envs shard).
Workload (config.workload): the C5 slice of BASELINE.json -- 131072 envs per GPU (1 Mi envs at 8
GPUs) x 1 LB agent x 64 servers, 128-slot reservoirs, synthetic Poisson flows (128 flows/s per
agent, rho=0.8), random policy.  A "step" is one launch of step_kernel over all envs of the rank.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
# A NCCL_DEBUG level the caller exported is left alone (its output goes wherever the caller pointed it).  Otherwise
# NCCL logs at INFO into a file, so that stdout stays the one JSON line and the communicator evidence (nranks,
# NVLS / ring choice) can still be read afterwards.  The file goes to the temporary directory: the benchmark writes
# nothing into the source tree, which may be read-only.
if "NCCL_DEBUG" not in os.environ:
    os.environ["NCCL_DEBUG"] = "INFO"
    os.environ["NCCL_DEBUG_SUBSYS"] = os.environ.get("NCCL_DEBUG_SUBSYS", "INIT,ENV")
    if "NCCL_DEBUG_FILE" not in os.environ:
        os.environ["NCCL_DEBUG_FILE"] = os.path.join(tempfile.gettempdir(), "marllb_b200_nccl_%h_%p.log")
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (envs/GPU, agents, servers/agent, flows/s per agent, K)
    "c5": dict(envs=131072, agents=1, servers=64, rate=128.0, K=128),
    "c2": dict(envs=4096, agents=1, servers=16, rate=32.0, K=128),
    "c3env": dict(envs=16384, agents=2, servers=32, rate=128.0, K=128),
    # config C3: QMIX action selection for every (env, agent) fused with the env step (marllb_b200/rollout.py);
    # network sizes as wired by the reference driver (training_pipeline.py:171-185), clean obs layout (Sa*11)
    "c3": dict(envs=16384, agents=2, servers=32, rate=128.0, K=128, policy="qmix"),
    # config C4 (per-GPU slice): one SAC-GRU learner over 1024 envs x 256 servers, actor inference + env step +
    # one SAC update (batch 256, device replay) per step; with N > 1 the gradient buckets are all-reduced over NCCL
    "c4": dict(envs=1024, agents=1, servers=256, rate=512.0, K=128, policy="sac"),
    # the same work per step with the SAC update as a graph branch BESIDE the env step (SACRollout.capture(overlap=True):
    # the update's batch is drawn from the replay ring as it stood before this step's push)
    "c4p": dict(envs=1024, agents=1, servers=256, rate=512.0, K=128, policy="sac", overlap=True),
}
RHO = 0.8
DT = 0.25
TS_BYTES = 4  # float32 timestamps (src/vpp/lb/shm.h:23-25)


def algorithmic_bytes_per_agent_step(S, K, F, T=TS_BYTES, log=False, replay=False):
    """SURVEY.md 8(d): S*(2K(4+T)+92) + F*(8+2(4+T)+4[log]+8[replay]) + S*4 + 5."""
    return S * (2 * K * (4 + T) + 92) + F * (8 + 2 * (4 + T) + 4 * log + 8 * replay) + S * 4 + 5


def algorithmic_bytes_split(S, K, F, T=TS_BYTES):
    """The same formula split over the two kernels of a step (DESIGN.md 4):
    feature kernel = reservoirs read once for the statistics + the 10 feature columns of obs + reward + done;
    event kernel   = per-server scalar state r/w, n_flow_on column, arrivals, reservoir slot writes, actions."""
    feature = S * (2 * K * (4 + T) + 40) + 5
    return algorithmic_bytes_per_agent_step(S, K, F, T) - feature, feature


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line):
    NVML polled every few milliseconds from a thread (the timed region of the default run is ~0.1 s, too
    short for `nvidia-smi -lms`); `nvidia-smi` once as the fallback."""
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index, period_s=0.004):
        self.idx, self.period = gpu_index, period_s
        self.sm, self.reasons, self.mx = [], set(), None
        self._stop, self.t, self.nvml = threading.Event(), None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.idx]) if vis and vis.split(",")[self.idx].isdigit() else self.idx
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.bits = {"hw_slowdown": pynvml.nvmlClocksThrottleReasonHwSlowdown,
                         "hw_thermal_slowdown": pynvml.nvmlClocksThrottleReasonHwThermalSlowdown,
                         "sw_thermal_slowdown": pynvml.nvmlClocksThrottleReasonSwThermalSlowdown,
                         "sw_power_cap": pynvml.nvmlClocksThrottleReasonSwPowerCap}
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
        except Exception:
            self.nvml = None

    def _poll(self):
        nv = self.nvml
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for n, b in self.bits.items():
                    if r & b:
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(self.period)

    def _smi_once(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            out = subprocess.run(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                 capture_output=True, text=True, timeout=10).stdout.strip().splitlines()[0]
            f = [x.strip() for x in out.split(",")]
            self.sm.append(float(f[0]))
            self.mx = float(f[1])
            for n, v in zip(self.NAMES, f[2:6]):
                if v.lower().startswith("active"):
                    self.reasons.add(n)
        except Exception:
            pass

    def stop(self):
        if self.t is not None:
            self._stop.set()
            self.t.join(timeout=2)
        source = "nvml"
        if not self.sm:
            self._smi_once()              # still inside the bracket: the GPU has only just gone idle
            source = "nvidia-smi"
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["clock query unavailable"]}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.mx, "samples": len(self.sm),
                "reasons": sorted(self.reasons), "source": source}


def cpu_oracle_rate(wl, n_envs, burnin, budget_s, threads, arrivals=None, seed=77):
    """Time the CPU restatement of the same env step (oracle/flow_oracle.c, pthreads) on a bounded
    sample of envs of the same workload.  Returns (agent_steps_per_s, steps_timed, threads)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import flow_oracle as fo
    S, A = wl["servers"], wl["agents"]
    threads = threads or fo.max_threads()
    speeds = np.where(np.arange(S * A) % 2 == 0, 1.0, 2.0).astype(np.float32)
    mean_work = RHO * speeds[:S].sum() / wl["rate"]
    rng = np.random.RandomState(seed)
    horizon = (burnin + 400) * DT
    envs = []
    for e in range(n_envs):
        if arrivals is not None:
            streams = arrivals[e]
        else:
            streams = []
            for _ in range(A):
                n = int(wl["rate"] * horizon * 1.2) + 64
                t = np.cumsum(rng.exponential(1.0 / wl["rate"], n))
                t = t[t < horizon].astype(np.float32)
                streams.append({"time": t, "work": rng.exponential(mean_work, len(t)).astype(np.float32)})
        envs.append(fo.FlowEnv(A, S, speeds, streams, reservoir_k=wl["K"], max_steps=10 ** 9))
    acts = rng.randint(0, 3, (8, n_envs, S * A)).astype(np.int32)
    for k in range(burnin):
        fo.step_batch(envs, acts[k % 8], threads)
    t0 = time.perf_counter()
    steps = 0
    while steps < 400 - 1:
        fo.step_batch(envs, acts[steps % 8], threads)
        steps += 1
        if time.perf_counter() - t0 > budget_s and steps >= 3:
            break
    dt = time.perf_counter() - t0
    return n_envs * A * steps / dt, steps, threads


def run_reference(args):
    """--impl reference: the reference path's CPU implementation (oracle port; the reference has no
    flow-level step of its own, SURVEY 0.1) on all host threads, same config/metric/unit."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import flow_oracle as fo
    threads = fo.max_threads()
    n_envs = max(threads * 4, 32)
    # K timed steps + W warm-up on the sample, after the same burn-in as the GPU arm
    S, A = wl["servers"], wl["agents"]
    speeds = np.where(np.arange(S * A) % 2 == 0, 1.0, 2.0).astype(np.float32)
    mean_work = RHO * speeds[:S].sum() / wl["rate"]
    rng = np.random.RandomState(77)
    total = args.burnin + args.warmup + args.steps
    horizon = (total + 2) * DT
    envs = []
    for e in range(n_envs):
        streams = []
        for _ in range(A):
            n = int(wl["rate"] * horizon * 1.2) + 64
            t = np.cumsum(rng.exponential(1.0 / wl["rate"], n))
            t = t[t < horizon].astype(np.float32)
            streams.append({"time": t, "work": rng.exponential(mean_work, len(t)).astype(np.float32)})
        envs.append(fo.FlowEnv(A, S, speeds, streams, reservoir_k=wl["K"], max_steps=10 ** 9))
    acts = rng.randint(0, 3, (8, n_envs, S * A)).astype(np.int32)
    for k in range(args.burnin + args.warmup):
        fo.step_batch(envs, acts[k % 8], threads)
    t0 = time.perf_counter()
    for k in range(args.steps):
        fo.step_batch(envs, acts[k % 8], threads)
    dt = time.perf_counter() - t0
    value = n_envs * A * args.steps / dt
    sample = f"{n_envs} envs x {A} agent x {S} servers, {args.steps} steps after {args.burnin}+{args.warmup} untimed"
    print(json.dumps({
        "impl": "reference", "metric": "agent-steps/sec", "value": value, "unit": "agent-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, wl),
        "cpu_baseline": {"value": value, "unit": "agent-steps/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def workload_config(args, wl, world=None, name=None):
    pol = {"qmix": "QMIX epsilon-greedy action selection (eps=0.05) fused with the env step",
           "sac": "SAC-GRU actor sampling + env step + one SAC update (batch 256) per step"
                  + (" (update pipelined beside the env step)" if wl.get("overlap") else ""),
           None: "random policy"}[wl.get("policy")]
    return {"workload": f"{name or args.workload}: {wl['envs']} envs/GPU x {wl['agents']} LB agent x {wl['servers']} servers, "
                        f"K={wl['K']}-slot reservoirs, Poisson {wl['rate']:.0f} flows/s/agent, rho={RHO}, {pol}, SED",
            "envs_per_gpu": wl["envs"], "agents": wl["agents"], "servers_per_agent": wl["servers"],
            "reservoir_k": wl["K"], "flows_per_s_per_agent": wl["rate"], "dt_s": DT,
            "burnin_steps": args.burnin,
            "l2_policy": "per-step working set (>17 GB of reservoirs per GPU) far exceeds the 126 MB L2",
            "parallelism": (f"env-sharded x{world or args.gpus}: no data-path collective in the env step"
                            + ("; SAC gradient buckets all-reduced over NCCL (captured in the step's CUDA graph)"
                               if wl.get("policy") == "sac" else ""))}


def build_env(wl, total_steps, rank=0, local=0, feature_cache=True, rng_mode="replay"):
    """The benchmarked env, exactly: used by run_ours and by tests/test_gpu_bench_parity.py (which steps THIS env and
    feeds sampled envs' device-generated arrivals to the CPU oracle).  Returns (env, speeds, action pool, generator)."""
    import torch
    from marllb_b200 import VecLoadBalanceEnv
    E, A, S, K = wl["envs"], wl["agents"], wl["servers"], wl["K"]
    env = VecLoadBalanceEnv(E, num_servers=S, num_agents=A, reservoir_capacity=K, max_steps=10 ** 9,
                            action_type="continuous" if wl.get("policy") == "sac" else "discrete",
                            action_dtype="uint8", env_id_base=rank * E, device=local,
                            feature_cache=feature_cache, rng_mode=rng_mode)
    speeds = np.where(np.arange(S * A) % 2 == 0, 1.0, 2.0).astype(np.float32)
    env.set_speeds(speeds)
    mean_work = RHO * float(speeds[:S].sum()) / wl["rate"]
    env.gen_poisson(wl["rate"], mean_work, (total_steps + 1) * DT, seed=1234)
    env.reset()
    g = torch.Generator(device="cuda")
    g.manual_seed(99 + rank)
    pool = [torch.randint(0, 3, (E, S * A), generator=g, device="cuda", dtype=torch.uint8) for _ in range(8)]
    return env, speeds, pool, g


def _setup_policy(wl, env, rank, local, gen):
    """QMIX (c3) / SAC (c4) rollouts on top of the env; returns (rollout, sac, draw pools)."""
    import torch
    E, A, S = wl["envs"], wl["agents"], wl["servers"]
    rollout = sac = sac_agent = None
    upool = rpool = None
    if wl.get("policy") == "qmix":
        from marllb_b200.policy import QMIXAgent
        from marllb_b200.rollout import QMIXRollout
        torch.manual_seed(7)   # random-init weights of the reference architecture
        agent = QMIXAgent(num_agents=A, state_dim=4 * A * S + 10, obs_dim=S * 11, action_dim=S, hidden_dim=64, gru_dim=64,
                          mixing_embed_dim=32, hypernet_embed_dim=64, device=torch.device("cuda", local))
        rollout = QMIXRollout(env, agent)
        upool = [torch.rand((E, A), generator=gen, device="cuda") for _ in range(8)]
        rpool = [torch.randint(0, S, (E, A), generator=gen, device="cuda", dtype=torch.int32) for _ in range(8)]
    if wl.get("policy") == "sac":
        from marllb_b200.policy import SAC_GRU_Agent
        from marllb_b200.rollout import SACRollout
        torch.manual_seed(7)   # same initial weights on every rank
        sac_agent = SAC_GRU_Agent(state_dim=S * 11, action_dim=S, hidden_dim=256, gru_dim=128, batch_size=256,
                                  device=torch.device("cuda", local))
        sac = SACRollout(env, sac_agent)
    return rollout, sac, sac_agent, upool, rpool


DUMP_ROWS_BYTES = 48 << 20   # per-env rows kept by --dump-outputs; with the rest the dump stays under 64 MB


def dump_outputs(out_dir, last, E):
    """--dump-outputs: what the last timed step returned to its caller, one <out_dir>/<name>.npy per array (float64
    stays float64, everything else becomes float32), so that two builds run with the same arguments can be compared
    output for output.  Arrays with one row per env keep a fixed, seeded sample of rows when all of them would exceed
    DUMP_ROWS_BYTES (c5: 131072 envs x 64 servers x 11 floats of observations); env_index.npy lists the rows kept.
    With N > 1 GPUs rank 0 writes its own shard of envs."""
    import torch
    step_out, losses = last if isinstance(last[0], tuple) else (last, None)      # SAC: ((obs, ...), losses)
    arrays = dict(zip(("obs", "reward", "done", "actions"), step_out))
    for k, v in (losses or {}).items():
        arrays[f"loss_{k}"] = v if isinstance(v, torch.Tensor) else torch.tensor(float(v), dtype=torch.float64)
    per_env = [v for v in arrays.values() if v.dim() and v.shape[0] == E]
    row_bytes = 8 + sum((8 if v.dtype == torch.float64 else 4) * (v.numel() // E) for v in per_env)
    rows = np.arange(E) if E * row_bytes <= DUMP_ROWS_BYTES else \
        np.sort(np.random.RandomState(0).choice(E, DUMP_ROWS_BYTES // row_bytes, replace=False))
    torch.cuda.synchronize()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "env_index.npy"), rows.astype(np.float64))
    for name, v in arrays.items():
        if v.dim() and v.shape[0] == E:
            v = v.index_select(0, torch.as_tensor(rows, device=v.device))
        v = v.detach().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), v if v.dtype == np.float64 else v.astype(np.float32))


def measure(args, name, world, rank, local, main):
    """One workload at N = world GPUs: burn-in, K timed steps (CUDA events, barrier + synchronize on both sides, max over
    ranks), per-kernel CUDA events; for the main workload also the end-to-end leg through host buffers and a second
    timed window late in the episode.  Returns the result dict on rank 0 (None elsewhere)."""
    import torch
    import torch.distributed as dist
    from marllb_b200.policy import ops as pops

    wl = dict(WORKLOADS[name])
    if args.envs and main:
        wl["envs"] = args.envs
    E, A, S, K = wl["envs"], wl["agents"], wl["servers"], wl["K"]
    steps, warmup = (args.steps, args.warmup) if main else (args.config_steps, max(3, args.warmup))
    burnin = args.burnin if main else min(args.burnin, args.config_burnin)
    e2e_steps = min(steps, args.e2e_steps) if main else 0
    late = main and args.late_burnin > burnin and wl.get("policy") is None
    total_steps = burnin + warmup + steps + 20 + e2e_steps + 24
    env, speeds, pool, g = build_env(wl, total_steps, rank, local, not args.no_feature_cache, args.rng_mode)
    mean_work = RHO * float(speeds[:S].sum()) / wl["rate"]
    rollout, sac, sac_agent, upool, rpool = _setup_policy(wl, env, rank, local, g)
    has_policy = rollout is not None or sac is not None
    sac_gen = None
    if sac is not None:
        sac_gen = torch.Generator(device="cuda")
        sac_gen.manual_seed(5 + rank)
    graphed = False

    def cur_step():
        return int(env.get_state("step", envs=[0])[0])      # steps the envs have taken (device counter, env.py:230)

    def do_step(k):
        """One step of the workload; returns what the path returns to its caller."""
        if sac is not None:
            if graphed:
                return sac.step_graph()
            out = sac.step()
            return out, sac.update(1, sac_gen)
        elif rollout is None and graphed:
            env.graph_action.copy_(pool[k % 8])
            return env.step_graph()
        elif rollout is None:
            return env.step(pool[k % 8])
        elif graphed:
            rollout.graph_u.copy_(upool[k % 8])
            rollout.graph_rnd.copy_(rpool[k % 8])
            return rollout.step_graph()
        else:
            return rollout.step(0.05, upool[k % 8], rpool[k % 8])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def launches_now():
        return env.launch_count + (pops.LAUNCHES if has_policy else 0)

    for k in range(burnin):
        do_step(k)
    prof_eager = None
    if rollout is not None and not args.no_graph:
        # per-kernel times of the env kernels from a short eager pass (event records are not captured),
        # then the whole rollout step as ONE CUDA-graph launch for the timed region
        env.profile_begin(10)
        for k in range(10):
            do_step(k)
        prof_eager = env.profile_end()
        rollout.capture(0.05)
        graphed = True
    env_graph = False
    if not main and not has_policy and not args.no_graph and E * A < 32768:
        # small batches are launch-gap bound (c2: 4096 warps = 0.7 of a wave): per-kernel times from a short eager
        # pass, then the four launches of a step replayed as one CUDA graph
        env.profile_begin(10)
        for k in range(10):
            do_step(k)
        prof_eager = env.profile_end()
        env.capture()
        env_graph = graphed = True
    if sac is not None and not args.no_graph:
        n_fill = 0
        while len(sac.replay) < sac.replay.capacity:      # the graph samples from a full ring
            do_step(0)
            n_fill += 1
        # a full ring costs capacity / E steps of simulated time: fresh arrivals from here on
        c0 = cur_step()
        env.gen_poisson(wl["rate"], mean_work, (c0 + warmup + steps + 64) * DT, seed=1234, t_start=c0 * DT, window=1)
        env.profile_begin(10)
        for k in range(10):
            do_step(k)
        prof_eager = env.profile_end()
        sac.capture(1, overlap=bool(wl.get("overlap")))   # under data parallelism the NCCL all-reduces are captured with it
        graphed = True

    def timed_window(n_steps):
        for k in range(warmup):
            do_step(k)
        env.check_status()
        cur0 = env.get_state("arr_cursor").astype(np.int64).sum()
        l0 = launches_now()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        env.profile_begin(n_steps)   # CUDA events around each kernel, on the launching stream
        barrier()
        ev0.record()
        last = None
        for k in range(n_steps):
            last = do_step(k)
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        prof = env.profile_end()
        pair_ms = getattr(env, "last_pair_ms", 0.0)
        n_launch = launches_now() - l0
        flows = env.get_state("arr_cursor").astype(np.int64).sum() - cur0
        env.check_status()
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        fl = torch.tensor([float(flows)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(fl, op=dist.ReduceOp.SUM)
        return float(t.item()), ms, prof, pair_ms, n_launch, float(fl.item()), last

    clocks = ClockSampler(local)
    if rank == 0 and main:
        clocks.start()
    ms_max, ms, prof, pair_ms, launches, flows, last = timed_window(steps)
    clk = clocks.stop() if (rank == 0 and main) else None
    if main and rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last, E)
    ev_ms, ft_ms, prof_steps = prof
    if prof_eager is not None:
        ev_ms, ft_ms, prof_steps = prof_eager
        pair_ms = None
    if graphed:
        launches = (env if env_graph else (rollout if rollout is not None else sac)).graph_launches * steps
    value = world * E * A * steps / (ms_max * 1e-3)

    # C4: the replicas must stay in lock-step (identical initial weights + identical averaged gradients): checksum of
    # every parameter, max - min over the ranks
    param_spread = None
    if sac_agent is not None:
        cs = torch.stack([b.flat_p.double().sum() for b in (sac_agent.policy_optimizer.bucket, sac_agent.q1_optimizer.bucket,
                                                          sac_agent.q2_optimizer.bucket)]).sum().reshape(1)
        hi, lo = cs.clone(), cs.clone()
        if world > 1:
            dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        param_spread = float((hi - lo).item())

    peak, which = measured_peaks()
    F = flows / (world * E * A * steps)
    bytes_as = algorithmic_bytes_per_agent_step(S, K, F)   # S = servers per agent
    b_event, b_stats = algorithmic_bytes_split(S, K, F)
    step_s = ms * 1e-3 / steps
    env_s = (ev_ms + ft_ms) * 1e-3 / max(prof_steps, 1)     # env kernels only (== step_s without a policy)
    res = {"value": value, "ms_per_step": ms_max / steps, "steps": steps, "burnin_steps": burnin,
           "flows_per_agent_step": F, "gpu_launches": int(launches), "cuda_graph": graphed,
           "env_kernels_ms": env_s * 1e3,
           "roofline_step": {"algorithmic_bytes_per_agent_step": bytes_as,
                             "achieved": bytes_as * E * A / env_s / 1e9, "frac": bytes_as * E * A / env_s / 1e9 / peak,
                             "of": "env-step kernels (event + statistics pass)"}}
    if has_policy:
        res["policy_ms_per_step"] = (step_s - env_s) * 1e3
    if param_spread is not None:
        res["param_checksum_spread_over_ranks"] = param_spread
    if not main:
        _release(env, rollout, sac)
        del env, rollout, sac, sac_agent, pool
        torch.cuda.empty_cache()
        return res if rank == 0 else None

    # ---- end to end through the public API with HOST buffers
    e2e_changed = None
    if has_policy:
        # what a trainer exchanges with the device-resident rollout per step: exploration draws in (pinned H2D),
        # rewards / dones (/ chosen actions) out (pinned D2H); observations stay on the device
        o_rew = torch.empty((E,), dtype=torch.float64, pin_memory=True)
        o_done = torch.empty((E,), dtype=torch.uint8, pin_memory=True)
        if sac is not None:
            h_eps = [torch.randn((E, S), dtype=torch.float32).pin_memory() for _ in range(2)]
            d_eps = torch.empty((E, S), dtype=torch.float32, device="cuda")

            def e2e_step(k):
                d_eps.copy_(h_eps[k % 2], non_blocking=True)
                if graphed:
                    (_, r_, dn_, _), _ = sac.step_graph()   # (Gaussian draws come from the device generator here)
                else:
                    _, r_, dn_, _ = sac.step(eps=d_eps)
                    sac.update(1, sac_gen)
                o_rew.copy_(r_, non_blocking=True)
                o_done.copy_(dn_, non_blocking=True)
                torch.cuda.current_stream().synchronize()
            h2d, e2e_d2h = E * S * 4, E * 8 + E
        else:
            h_u = [torch.empty((E, A), dtype=torch.float32, pin_memory=True).copy_(upool[i]) for i in range(2)]
            h_r = [torch.empty((E, A), dtype=torch.int32, pin_memory=True).copy_(rpool[i]) for i in range(2)]
            d_u, d_r = torch.empty_like(upool[0]), torch.empty_like(rpool[0])
            o_act = torch.empty((E, A), dtype=torch.int32, pin_memory=True)

            def e2e_step(k):
                if graphed:
                    rollout.graph_u.copy_(h_u[k % 2], non_blocking=True)
                    rollout.graph_rnd.copy_(h_r[k % 2], non_blocking=True)
                    _, r_, dn_, a_ = rollout.step_graph()
                else:
                    d_u.copy_(h_u[k % 2], non_blocking=True)
                    d_r.copy_(h_r[k % 2], non_blocking=True)
                    _, r_, dn_, a_ = rollout.step(0.05, d_u, d_r)
                o_rew.copy_(r_, non_blocking=True)
                o_done.copy_(dn_, non_blocking=True)
                o_act.copy_(a_, non_blocking=True)
                torch.cuda.current_stream().synchronize()
            h2d, e2e_d2h = E * A * 8, E * 8 + E + E * A * 4
        torch.cuda.synchronize()
        e2e_step(0)
        barrier()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            e2e_step(k)
        torch.cuda.synchronize()
        te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_value = world * E * A * e2e_steps / float(te.item())
        e2e_api = "device-resident rollout: exploration draws in, rewards / dones / actions out per step"
    else:
        h_act = []
        for p_ in pool[:2]:
            t_ = env.pinned_actions()
            t_.copy_(p_.view_as(t_))
            h_act.append(t_)
        torch.cuda.synchronize()

        def e2e_leg(mode):
            env.step_host(h_act[0], obs=mode)  # allocates pinned output buffers / builds the host mirror, untimed
            barrier()
            t0 = time.perf_counter()
            moved = 0
            for k in range(e2e_steps):
                env.step_host(h_act[k % 2], obs=mode)
                moved += env.last_d2h_bytes
            torch.cuda.synchronize()
            te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            return world * E * A * e2e_steps / float(te.item()), moved / max(e2e_steps, 1)

        e2e_value, e2e_d2h = e2e_leg("full")
        e2e_changed = e2e_leg("changed")
        h2d = env.e2e_bytes[0]
        e2e_api = "VecLoadBalanceEnv.step_host(actions): full (E,S,11) float32 observations into pinned host memory"

    # ---- second timed window, late in the episode (acceptance of Algorithm R ~ K / count: few touched reservoirs)
    late_res = None
    if late:
        chunk, win = 448, 1
        while True:
            c0 = cur_step()
            if c0 >= args.late_burnin:
                break
            n = min(chunk, args.late_burnin - c0)
            tail = warmup + steps + 4 * (e2e_steps + 1) + 8 if c0 + n >= args.late_burnin else 0
            env.gen_poisson(wl["rate"], mean_work, (c0 + n + tail) * DT, seed=1234, t_start=c0 * DT, window=win)
            win += 1
            for k in range(n):
                do_step(k)
        l_ms_max, l_ms, l_prof, l_pair, _, l_flows, _ = timed_window(steps)
        l_ev, l_ft, l_n = l_prof
        l_F = l_flows / (world * E * A * steps)
        l_bytes = algorithmic_bytes_per_agent_step(S, K, l_F)
        late_res = {"burnin_steps": args.late_burnin, "ms_per_step": l_ms_max / steps,
                    "value": world * E * A * steps / (l_ms_max * 1e-3),
                    "event_kernel_ms": l_ev / max(l_n, 1), "statistics_pass_ms": l_ft / max(l_n, 1),
                    "pair_kernel_ms": l_pair / max(l_n, 1), "flows_per_agent_step": l_F,
                    "algorithmic_frac": l_bytes * E * A / (l_ms * 1e-3 / steps) / 1e9 / peak,
                    "note": "most reservoirs are untouched in a step this deep into an episode and are not re-read, "
                            "so the algorithmic fraction (all reservoirs re-read) overstates DRAM use; the event "
                            "kernel dominates here"}
        e2e_late_full = e2e_leg("full")
        e2e_late = e2e_leg("changed")
        late_res["e2e"] = {"value": e2e_late_full[0], "d2h_bytes_per_step": e2e_late_full[1],
                           "changed_rows": {"value": e2e_late[0], "d2h_bytes_per_step": e2e_late[1]}}

    if rank != 0:
        return None
    ft_avg_s = ft_ms * 1e-3 / max(prof_steps, 1)
    ev_avg_s = ev_ms * 1e-3 / max(prof_steps, 1)
    pr_avg_s = (pair_ms or 0.0) * 1e-3 / max(prof_steps, 1)
    traffic = tsrc = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            tj = json.load(f)
        traffic, tsrc = tj.get(name, {}), tj.get("_source")
    phys_step = (traffic.get("statistics_pass_total", 0) + traffic.get("event_kernel", 0)) if traffic else None
    step_achieved = bytes_as * E * A / step_s / 1e9
    res.update({
        "roofline": {
            "bound": "hbm", "achieved": step_achieved, "peak": peak, "unit": "GB/s", "frac": step_achieved / peak,
            "peak_source": which,
            "kernel": "whole env step = mlb::event_kernel + mlb::pair_kernel<.,0> + mlb::pair_kernel<.,1> + "
                      "mlb::feature_kernel (four launches); headline frac = algorithmic bytes of the step / step time",
            "algorithmic_bytes_per_agent_step": bytes_as,
            # NOT sampled in this run: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of
            # the same command, per launch, committed under profiles/ (see traffic_source)
            "traffic": phys_step, "traffic_source": tsrc,
            "physical": ({"achieved": phys_step / step_s / 1e9, "frac": phys_step / step_s / 1e9 / peak,
                          "note": "profiled DRAM bytes (profiles/traffic.json) over THIS run's step time"}
                         if phys_step else None),
            "kernels": [
                {"kernel": "mlb::event_kernel<SED>", "ms": ev_avg_s * 1e3, "algorithmic_bytes_per_agent_step": b_event,
                 "achieved": b_event * E * A / ev_avg_s / 1e9 if ev_avg_s > 0 else None,
                 "traffic": traffic.get("event_kernel") if traffic else None, "bound": "issue / latency"},
                {"kernel": "statistics pass: mlb::pair_kernel x2 + mlb::feature_kernel (three launches)",
                 "ms": ft_avg_s * 1e3, "pair_kernels_ms": pr_avg_s * 1e3,
                 "algorithmic_bytes_per_agent_step": b_stats,
                 "achieved": b_stats * E * A / ft_avg_s / 1e9, "frac": b_stats * E * A / ft_avg_s / 1e9 / peak,
                 "traffic": traffic.get("statistics_pass_total") if traffic else None,
                 "physical_frac": (traffic["statistics_pass_total"] / ft_avg_s / 1e9 / peak) if traffic and traffic.get("statistics_pass_total") else None,
                 "note": "the algorithmic fraction can exceed 1: reservoirs untouched in a step keep their cached features "
                         "and are not re-read (SURVEY 8d asks for both numbers)", "bound": "hbm"}],
            "kernel_share_of_step": {"event": ev_ms / max(ft_ms + ev_ms, 1e-9), "statistics": ft_ms / max(ft_ms + ev_ms, 1e-9)},
            "flows_per_agent_step": F, "late_episode": late_res},
        "e2e": {"value": e2e_value, "unit": "agent-steps/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": e2e_d2h, "steps": e2e_steps, "api": e2e_api,
                "changed_rows": ({"value": e2e_changed[0], "d2h_bytes_per_step": e2e_changed[1],
                                  "api": "step_host(actions, obs='changed'): n_flow_on column + only the rows in which a "
                                         "reservoir slot was written, applied by host threads to the persistent host "
                                         "observation array (bit-equal result)"} if e2e_changed else None)},
        "clocks": clk})
    _release(env, rollout, sac)
    del env, pool
    torch.cuda.empty_cache()
    return res


def _release(env, rollout, sac):
    """CUDA graphs that hold NCCL kernels must be gone before the process group is torn down (a communicator destroyed
    under a live graph hangs at exit): reset every captured graph, then free the env."""
    import gc
    import torch
    torch.cuda.synchronize()
    for obj in (env, rollout, sac):
        g = getattr(obj, "_graph", None)
        if g is not None:
            g.reset()
            obj._graph = None
    env.close()
    gc.collect()
    torch.cuda.synchronize()


def cpu_legs(args, wl):
    """CPU numbers reported beside the GPU line (BASELINE.md section 3): (ii) the C restatement of the composed flow
    env on all host threads = `cpu_baseline`; (iii) the reference's own C reservoir micro-benchmark (oracle/_ref, built
    from the reference's reservoir.c by oracle/Makefile: a native upper bound for one add); (i) the reference's literal
    simulation-mode step (random features + reward, env.py:215-286) through its C restatement on all threads."""
    import re
    n_envs = max(4 * (os.cpu_count() or 1), 32)
    v, steps, cores = cpu_oracle_rate(wl, n_envs=n_envs, burnin=args.burnin, budget_s=args.cpu_budget, threads=0)
    out = {"value": v, "unit": "agent-steps/s", "cores": cores, "kind": "port",
           "sample": f"{n_envs} envs of the same workload, {steps} steps after {args.burnin} burn-in steps, "
                     f"oracle/flow_oracle.c on {cores} threads",
           "note": "a LITERAL port of the reference's Python arithmetic (every touched reservoir re-sorted, float64 pow "
                   "per slot), as the parity oracle must be: a baseline for orientation, not an optimised CPU program"}
    exe = os.path.join(ROOT, "oracle", "_ref", "reservoir_c_bench")
    if os.path.exists(exe):
        try:
            txt = subprocess.run([exe], capture_output=True, text=True, timeout=60).stdout
            m = re.search(r"Throughput:\s*([0-9.]+)\s*M ops/sec", txt)
            if m:
                out["reference_c_reservoir_add"] = {"value": float(m.group(1)) * 1e6, "unit": "adds/s", "cores": 1,
                                                    "kind": "reference",
                                                    "what": "reference's reservoir.c benchmark (reservoir.c:77-102), unmodified"}
        except Exception as exc:   # noqa: BLE001
            out["reference_c_reservoir_add"] = {"unavailable": str(exc)}
    try:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import flow_oracle as fo
        S = wl["servers"] * wl["agents"]
        t0, n = time.perf_counter(), 0
        g = fo.LegacyObs(1)
        while time.perf_counter() - t0 < 1.0:
            for _ in range(200):
                fo.reward_from_obs("jain", 10, g.next(S))
            n += 200
        out["reference_literal_step"] = {"value": n / (time.perf_counter() - t0), "unit": "env-steps/s", "cores": 1,
                                         "kind": "port", "what": "what LoadBalanceEnv.step literally does in simulation "
                                         "mode (env.py:425-448 random features + reward), C restatement, one thread; "
                                         "the Python original: 681 steps/s at 64 servers (BASELINE.md)"}
    except Exception as exc:       # noqa: BLE001
        out["reference_literal_step"] = {"unavailable": str(exc)}
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    # host side of the end-to-end step: pinned buffers on the NUMA node next to this rank's GPU
    from marllb_b200.shard import bind_host_to_gpu
    prev_affinity = bind_host_to_gpu(local) if (world > 1 and not os.environ.get("MLB_NO_NUMA_BIND")) else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    wl = dict(WORKLOADS[args.workload])
    res = measure(args, args.workload, world, rank, local, main=True)
    configs = {}

    def emit():
        """The ONE JSON line (rank 0), from whatever has been measured so far."""
        out = {
            "metric": "agent-steps/sec", "value": res["value"], "unit": "agent-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args, wl, world),
            "roofline": res["roofline"], "e2e": res["e2e"], "gpu_launches": res["gpu_launches"], "clocks": res["clocks"],
        }
        if configs:
            # the other BASELINE.json configurations at the same N (short runs; c4 is the one with a collective:
            # SAC update sharded over the GPUs, NCCL all-reduce of the gradient buckets inside the CUDA graph)
            out["configs"] = dict(configs)
        if world > 1:
            out["nccl"] = {"nranks": world, "version": ".".join(map(str, torch.cuda.nccl.version())),
                           "debug": os.environ.get("NCCL_DEBUG"), "log": os.environ.get("NCCL_DEBUG_FILE")}
        return out

    if not args.no_configs and args.workload == "c5":
        # dead-man switch for the side configurations: they must never cost the headline line.  If one of them does
        # not come back (a collective that hangs on a sick link, say) the line goes out without it and every rank exits.
        current = {"name": None}

        def give_up():
            if rank == 0:
                configs[current["name"]] = {"error": f"did not finish within {args.config_deadline:.0f} s; skipped"}
                print(json.dumps(emit()))
                sys.stdout.flush()
            os._exit(0)

        for name in ("c2", "c3", "c4", "c4p"):
            current["name"] = name
            dog = threading.Timer(args.config_deadline, give_up)
            dog.daemon = True
            dog.start()
            r = measure(args, name, world, rank, local, main=False)
            dog.cancel()
            if rank == 0:
                r["config"] = workload_config(args, WORKLOADS[name], world, name)["workload"]
                configs[name] = r
    if rank == 0:
        out = emit()
        if world == 1 and not args.no_cpu and wl.get("policy") is None:
            if prev_affinity is not None:
                os.sched_setaffinity(0, prev_affinity)       # the CPU baseline uses every host core
            out["cpu_baseline"] = cpu_legs(args, wl)
        print(json.dumps(out))
    sys.stdout.flush()
    if world > 1:
        # dead-man switch: the JSON line is out; a teardown that does not finish (seen with NCCL kernels captured in CUDA
        # graphs) must not keep the launcher waiting
        t = threading.Timer(20.0, lambda: os._exit(0))
        t.daemon = True
        t.start()
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()
        t.cancel()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c5", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=0, help="override envs per GPU")
    ap.add_argument("--burnin", type=int, default=256, help="untimed steps that bring reservoirs to steady state")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--late-burnin", type=int, default=2048,
                    help="second timed window after this many steps of the episode (0: skip)")
    ap.add_argument("--no-configs", action="store_true", help="skip the short c2 / c3 / c4 runs of the `configs` sub-dict")
    ap.add_argument("--config-steps", type=int, default=30)
    ap.add_argument("--config-burnin", type=int, default=256)
    ap.add_argument("--config-deadline", type=float, default=150.0,
                    help="seconds after which a side configuration (c2 / c3 / c4) is abandoned and the line printed without it")
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-feature-cache", action="store_true")
    ap.add_argument("--rng-mode", default="replay", choices=["replay", "philox"],
                    help="reservoir index stream: replayed RandomState rows shared by all envs (reference parity) "
                         "or per-env counter-based Philox")
    ap.add_argument("--no-graph", action="store_true", help="c3: launch the rollout step eagerly instead of as a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (obs, reward, done, ...) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
