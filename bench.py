#!/usr/bin/env python
"""bench.py -- the hot path's headline benchmark (BASELINE.json: env steps/sec + DQN updates/sec,
500x500x100 city) on N B200s of one node, with the reference's CPU path timed beside it.

One "step" = one lockstep training iteration of the workload: every env does
    state -> eps-greedy Q-net action -> UAV step (kinematics, collision, reward, termination,
    100-d observation) -> replay add
followed by ONE DQN update (sample B transitions, TD target, MSE, backward, Adam, periodic hard
target update) -- PathPlan_City.run_thread_OffPolicy + update (Envs/PathPlan_City.py:364-385,757-776).

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference ...                     (the CPU arm: the oracle port on the host threads)
  python bench.py ... --dump-outputs DIR                   (also write what the last timed step computed, DIR/<name>.npy)

Prints ONE JSON line (rank 0).
  value      whole-job env steps/s, inputs resident in HBM.  After W warm-up steps, exactly K steps are timed as one block
             (barrier + synchronize on both sides, CUDA events, max over ranks); the default K makes that window about 1 s on
             one B200 at the default workload.  --dump-outputs writes the state right after this block, before anything below
             runs, so it depends on the arguments alone.  The measurements below keep their own bounded step counts.
  e2e        the same iteration through the reference-facing plug-in classes (PathPlan_City_B200 / DQN_Trainer_B200 built
             from the XML configs) with HOST arrays at every boundary, H2D/D2H inside the timed region.
  roofline   dominant kernel: algorithmic bytes|flops / CUDA-event time vs MEASURED_PEAKS.json.
  cpu_baseline  the oracle port on the host cores (bounded sample) + the Python reference's own measured figure as context.
  configs    sub-results for the other BASELINE configs that fit this launch (N=1: 16 384-env DuelingDQN and SAC; N=8: 65 536-env DDQN).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

OBS = 100
NETS = {"qvalue3": ([64, 64], 0), "qnet2": ([64], 0), "vanet2": ([64], 1), "vanet3": ([128, 64], 1)}
NET_XML = {"qvalue3": "QValueNet_SAC", "qnet2": "Qnet2", "vanet2": "VAnet2", "vanet3": "VAnet3"}
ALGOS = {"dqn": 0, "ddqn": 1, "dueling": 2}
TRAINER_XML = {"dqn": "DQN_Trainer_B200", "ddqn": "DDQN_Trainer_B200", "dueling": "DuelingDQN_Trainer_B200"}
# SURVEY.md section 8(d): algorithmic bytes / flops per unit
ENV_STEP_BYTES = 563            # per env step (discrete action): obs 400 + reward 4 + flags 3 + action 4 + state r/w 128 + sub-goals 24
ACT_BYTES = 404                 # per env: obs read 400 + action write 4
TRANSITION_BYTES = 812          # per sampled transition
FWD_FLOPS = {"qvalue3": 24448, "qnet2": 2 * (100 * 64 + 64 * 27), "vanet2": 2 * (100 * 64 + 64 * 28),
             "vanet3": 2 * (100 * 128 + 128 * 64 + 64 * 28)}
PYTHON_REFERENCE = {"value": 100.0, "unit": "env_steps/s", "cores": 1, "kind": "python_reference",
                    "sample": "the unmodified Python reference (simulator.StartAndTrain, shipped SAC config, render stubbed), measured at "
                              "survey time on one core of an 8-vCPU Xeon 2.1 GHz container (BASELINE.md / SURVEY.md section 6): ~100 env steps/s "
                              "with training, ~450 env-only; it is GIL-bound, cannot travel to the GPU box and is quoted as context only"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps of the headline loop (default 25000: about 1 s at 45 us per step on one B200; 200 with --impl reference)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=4096, help="envs per GPU (BASELINE configs[1])")
    ap.add_argument("--batch", type=int, default=0, help="DQN batch per GPU per update (0 = envs: one sample per generated transition)")
    ap.add_argument("--net", default="qvalue3", choices=list(NETS))
    ap.add_argument("--algo", default="dqn", choices=list(ALGOS))
    ap.add_argument("--replay", type=int, default=1 << 20, help="replay capacity per GPU (transitions)")
    ap.add_argument("--pool", type=int, default=2048, help="scenario pool size (host RRT)")
    ap.add_argument("--eps", type=float, default=0.1)
    ap.add_argument("--tc", type=int, default=1, help="1 = tcgen05 3xTF32 tensor-core path for the Q-network (default), 0 = fp32 CUDA cores")
    ap.add_argument("--dp", default="fused", choices=["fused", "nccl"],
                    help="N>1 gradient exchange: fused = one-shot NVLink all-reduce inside the Adam kernel, nccl = torch.distributed")
    ap.add_argument("--dp-self", type=int, default=0, help="diagnostic, 1 GPU only: run the data-parallel loop (local gradient -> all-reduce + Adam kernel) with world = 1")
    ap.add_argument("--pdl", type=int, default=1, help="1 = programmatic dependent launch inside the loop (default), 0 = fully serialised kernels")
    ap.add_argument("--fuse", type=int, default=0, help="1 = get_action + env step as one kernel on the tensor-core path, 0 = two PDL-chained kernels (default, faster)")
    ap.add_argument("--fuse-dw", type=int, default=-1, help="1 = optimiser step inside the weight-gradient kernel (uavrl_set_fuse_dw_adam), 0 = separate kernel, -1 = library default")
    ap.add_argument("--per", type=int, default=0, help="1 = prioritised replay (device SumTree equivalent) instead of uniform sampling")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the env state, observations and learner state of the last step as DIR/<name>.npy")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the sub-results for the other BASELINE configs")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--threads", type=int, default=0, help="CPU arm: host threads (0 = every CPU this process may run on)")
    return ap.parse_args()


def load_city():
    g = np.load(os.path.join(ROOT, "tests", "golden", "env_golden.npz"))
    return g["dims"], np.ascontiguousarray(g["buildings"]), g["uav_params"]


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tf=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons of ONE GPU every 20 ms, started before the timed region's first barrier."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, gpu_index):
        self.idx, self.p, self.path = gpu_index, None, "/tmp/uavrl_clocks_%d.csv" % os.getpid()

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def mark(self):
        """number of lines written so far (the sampler starts before the region; samples from here on are 'under load')"""
        try:
            self.f.flush()
            return sum(1 for _ in open(self.path))
        except Exception:
            return 0

    def stop(self, first_line=0):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.p:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.close()
        sm, mx, util, reasons = [], [], [], set()
        for i, line in enumerate(open(self.path)):
            if i < first_line:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
            try:
                util.append(float(f[8]))
            except (ValueError, IndexError):
                pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_min_mhz=min(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm),
                       gpu_util_median=(statistics.median(util) if util else None))
        try:
            os.remove(self.path)
        except OSError:
            pass
        return out


def config_dict(a, world):
    return {"workload": "%d parallel UAV envs per GPU x %d GPU, PathPlan_City 500x500x100, 26 cylinder buildings "
                        "(reference config/buildings.xml), discrete-27 actions, %s %s MLP 100-%s-27, batch %d/GPU, "
                        "1 update per lockstep step, replay %d transitions/GPU"
                        % (a.envs, world, a.algo.upper(), a.net, "-".join(map(str, NETS[a.net][0])), a.batch, a.replay),
            "envs_per_gpu": a.envs, "global_envs": a.envs * world, "batch_per_gpu": a.batch, "global_batch": a.batch * world,
            "net": a.net, "algo": a.algo, "replay_per_gpu": a.replay, "prioritised_replay": bool(getattr(a, "per", 0)), "eps": a.eps, "scenario_pool": a.pool,
            "parallelism": "dp%d (env shards + replay shards per GPU, %s)" % (world, "one-shot NVLink all-reduce fused into the Adam kernel" if a.dp == "fused" else "NCCL gradient all-reduce"),
            "l2": "replay ring %d MB/GPU > 126 MB L2, fully prefilled before timing; sampled rows come from all of it"
                  % (a.replay * 412 // 1000000)}


# ============================================================================ CPU arm (oracle port; never maps the product library)
_USABLE = None


def usable_cpus():
    """CPUs this process may actually run on: the affinity mask at start-up (an OpenMP runtime with OMP_PROC_BIND later pins
    the calling thread, which would shrink the mask seen from it), capped by a cgroup CPU quota if there is one
    (the GPU boxes show 128 logical CPUs under a 16-CPU cpu.max quota)."""
    global _USABLE
    if _USABLE is not None:
        return _USABLE
    n = len(os.sched_getaffinity(0))
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(p))))
    except (OSError, ValueError):
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // p))
        except (OSError, ValueError):
            pass
    _USABLE = n
    return n


def cpu_env(threads, bind):
    """Must run before liboracle.so (libgomp) is loaded: torchrun exports OMP_NUM_THREADS=1, which is not what the CPU arm is.
    bind: pin the oracle's threads (OMP_PROC_BIND) -- only in the CPU-arm process, where the oracle's libgomp is the only
    OpenMP runtime; in the GPU process torch's own runtime would pin the main thread to one CPU and starve the oracle."""
    n = threads if threads > 0 else usable_cpus()
    os.environ["OMP_NUM_THREADS"] = str(n)
    os.environ.setdefault("OMP_DYNAMIC", "false")
    if bind:
        os.environ.setdefault("OMP_PROC_BIND", "spread")
        os.environ.setdefault("OMP_PLACES", "threads")
    return n


def make_oracle_loop(a, n_envs, threads):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    nthreads = O.set_threads(threads if threads > 0 else usable_cpus())
    pool = np.load(os.path.join(ROOT, "oracle", "pool_512.npz"))        # committed scenarios (oracle/make_pool.py)
    dims, b, p = pool["dims"], np.ascontiguousarray(pool["buildings"]), pool["uav_params"]
    P = len(pool["n_sub"])
    sub = np.zeros((P, 64, 3)); sub[:, :pool["sub"].shape[1]] = pool["sub"]
    sc = dict(start=pool["start"], goal=pool["goal"], heading=pool["heading"], sub=sub, n_sub=pool["n_sub"])
    hidden, dueling = NETS[a.net]
    net = O.make_net(OBS, hidden, 27, dueling)
    rng = np.random.default_rng(0)
    params = (rng.uniform(-1, 1, O.net_param_count(net)) * 0.1).astype(np.float32)
    city = O.OracleCity(dims[0], dims[1], dims[2], b)
    par = O.UavParams(p[0], p[1], p[2], 1.0, int(p[3]))
    loop = O.OracleTrainLoop(city, par, sc, n_envs, net, ALGOS[a.algo], params, a.batch, max(8 * n_envs, 4 * a.batch))
    return loop, nthreads


def cpu_baseline(a, seconds):
    """The oracle port timed on the host cores: bounded sample of the same workload."""
    loop, nthreads = make_oracle_loop(a, a.envs, a.threads)
    loop.iteration(a.eps); loop.iteration(a.eps)                   # warm-up (fills the replay past Batch_Size)
    t0 = time.perf_counter(); it = 0
    while it < 3 or time.perf_counter() - t0 < seconds:
        loop.iteration(a.eps); it += 1
    dt = time.perf_counter() - t0
    return {"value": a.envs * it / dt, "unit": "env_steps/s", "updates_per_s": it / dt, "cores": nthreads,
            "kind": "port", "usable_cpus": usable_cpus(), "omp_proc_bind": os.environ.get("OMP_PROC_BIND"),
            "sample": "%d lockstep iterations (%d envs each + 1 %s update, batch %d) of the C oracle port "
                      "(oracle/*.c, OpenMP, %d threads) in %.1f s" % (it, a.envs, a.algo.upper(), a.batch, nthreads, dt),
            "python_reference": PYTHON_REFERENCE}


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    loop, nthreads = make_oracle_loop(a, a.envs, a.threads)
    for _ in range(max(a.warmup, 2)):
        loop.iteration(a.eps)
    t0 = time.perf_counter()
    for _ in range(a.steps):
        loop.iteration(a.eps)
    dt = time.perf_counter() - t0
    v = a.envs * a.steps / dt
    sample = ("each step = one lockstep iteration of %d envs + 1 %s update (batch %d) on the oracle port, %d OpenMP threads "
              "(C restatement of the Python reference; the Python reference itself cannot travel to the GPU box); "
              "%d timed steps" % (a.envs, a.algo.upper(), a.batch, nthreads, a.steps))
    out = {"impl": "reference", "metric": "env steps/sec (+ DQN updates/sec), 500x500x100 city", "value": v,
           "unit": "env_steps/s", "updates_per_s": a.steps / dt, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
           "timed_region_s": dt,
           "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f64 env / f32 learner", "data": "synthetic", "config": config_dict(a, 1),
           "cpu_baseline": {"value": v, "unit": "env_steps/s", "cores": nthreads, "kind": "port", "sample": sample,
                            "usable_cpus": usable_cpus(), "omp_proc_bind": os.environ.get("OMP_PROC_BIND"),
                            "python_reference": PYTHON_REFERENCE},
           "e2e": {"value": v, "unit": "env_steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out, default=float), flush=True)


# ============================================================================ GPU arm
class Workload:
    """env batch + learner of one BASELINE config on this rank's GPU, replay ring prefilled."""

    def __init__(self, a, rank, world, local, dist):
        import torch
        import uavrl_b200  # noqa: F401
        from uavrl_b200 import engine
        self.a, self.rank, self.world, self.dist, self.engine, self.torch = a, rank, world, dist, engine, torch
        dims, b, p = load_city()
        city = engine.City(dims[0], dims[1], dims[2], b)
        params = engine.UavParams(p[0], p[1], p[2], 1.0, int(p[3]))
        N, B = a.envs, a.batch
        self.env = engine.EnvBatch(city, params, N, max_subgoals=64, device=local, auto_reset=True)
        sc = self.env.make_scenarios(a.pool, seed=42 + rank)
        self.env.set_pool(sc["start"], sc["goal"], sc["heading"], sc["sub"], sc["n_sub"])
        self.env.reset(0)
        hidden, dueling = NETS[a.net]
        self.L = engine.Learner(OBS, hidden, 27, dueling, ALGOS[a.algo], lr=5e-4, gamma=0.99, batch_size=B, update_loop=3,
                                replay_capacity=a.replay, lockstep_envs=N, seed=1234 + rank, device=local)
        self.L.init_params(0)                       # same seed on every rank: replicas start identical
        if a.per:
            self.L.per_enable()
        self.tc_on = self.L.set_tensor_cores(bool(a.tc))
        if world > 1 and a.dp == "fused":
            self.L.connect_peers(dist, rank, world)
        elif world == 1 and a.dp_self:
            self.L.connect_self()
        ring_frames = (a.replay + N - 1) // N + 1
        engine.train_run(self.env, self.L, ring_frames, 1.0, 1, False, want_stats=False)     # prefill: sampling spans > L2 worth of rows

    def iterate(self, k):
        """k lockstep iterations.  1 GPU: the fused C loop.  N GPUs: env/act/ring per rank, local gradient, then the fused
        one-shot NVLink all-reduce + Adam (or NCCL all-reduce + Adam with --dp nccl), identical step on every rank."""
        a, engine = self.a, self.engine
        if self.world == 1 and a.dp_self:
            engine.train_run_dp(self.env, self.L, k, a.eps, a.batch)
        elif self.world == 1:
            engine.train_run(self.env, self.L, k, a.eps, 1, True, want_stats=False)
        elif a.dp == "fused":
            engine.train_run_dp(self.env, self.L, k, a.eps, a.batch * self.world)
        else:
            gt = self.L.grad_tensor()
            for _ in range(k):
                engine.train_run(self.env, self.L, 1, a.eps, 1, False, want_stats=False)
                self.L.compute_grads(a.batch * self.world)
                self.dist.all_reduce(gt, op=self.dist.ReduceOp.SUM)
                self.L.apply_grads()

    def close(self):
        self.L.close(); self.env.close()


def timed_steps(wl, a, dev, stream, barrier, sampler=None):
    """The K = --steps timed steps as one block: barrier + synchronize on both sides, CUDA events on the launching stream.
    Returns the block's ms (max over ranks), wall seconds of the region, sampler mark."""
    import torch
    world, dist = wl.world, wl.dist
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    mark = sampler.mark() if sampler else 0
    barrier()
    t0 = time.perf_counter()
    e0.record(stream)
    wl.iterate(a.steps)
    e1.record(stream)
    barrier()
    wall = time.perf_counter() - t0
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()), wall, mark


def dump_outputs(wl, out_dir, max_envs=1 << 16):
    """What a caller of the timed loop receives after its last step, as float32/float64 .npy files: this rank's env state
    (the step's reward, done flags, fp64 kinematics, counters) and observations, and the learner's parameters, Adam moments
    and last gradient.  Batches above max_envs are cut to a fixed seeded sample of envs (env_index.npy), which keeps the
    files well under 64 MB."""
    os.makedirs(out_dir, exist_ok=True)
    st = wl.env.get_state()
    st["obs"] = wl.env.observe().cpu().numpy()
    n = wl.env.n
    rows = np.arange(n) if n <= max_envs else np.sort(np.random.default_rng(0).choice(n, max_envs, replace=False))
    arrays = {"env_index": rows.astype(np.float64)}
    for k, v in st.items():
        v = v[rows]
        arrays["env_" + k] = v if v.dtype in (np.float32, np.float64) else v.astype(np.float64)
    for which, k in enumerate(("q_local", "q_target", "adam_exp_avg", "adam_exp_avg_sq", "grad")):
        arrays["learner_" + k] = wl.L.get_params(which)
    arrays["learner_counters"] = np.array(wl.L.counters(), np.float64)          # epoch, Adam step
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def measure_config(a_sub, rank, world, local, dist, dev, stream, barrier, label):
    """One sub-result (another BASELINE config) with the same timing discipline; returns a small dict (rank 0) or None."""
    wl = Workload(a_sub, rank, world, local, dist)
    wl.iterate(max(a_sub.warmup, 3))
    ms, wall, _ = timed_steps(wl, a_sub, dev, stream, barrier)
    out = {"label": label, "value": a_sub.envs * world * a_sub.steps / (ms * 1e-3), "unit": "env_steps/s",
           "updates_per_s": a_sub.steps / (ms * 1e-3), "ms_per_step": ms / a_sub.steps,
           "timed_region_s": wall, "n_gpus": world, "config": config_dict(a_sub, world), "tensor_cores": bool(wl.tc_on)}
    wl.close()
    return out if rank == 0 else None


def measure_sac(a, local, dev, stream, label):
    """BASELINE configs[4]: SAC continuous, 16 384 envs, 1 GPU."""
    import torch
    from uavrl_b200 import engine
    dims, b, p = load_city()
    city = engine.City(dims[0], dims[1], dims[2], b)
    params = engine.UavParams(p[0], p[1], p[2], 1.0, int(p[3]))
    N = 16384
    env = engine.EnvBatch(city, params, N, max_subgoals=64, device=local, auto_reset=True)
    sc = env.make_scenarios(a.pool, seed=42)
    env.set_pool(sc["start"], sc["goal"], sc["heading"], sc["sub"], sc["n_sub"])
    env.reset(0)
    L = engine.SacLearner(100, 64, 2, 1.0, 1e-4, 1e-3, 1e-4, 1.0, 0.99, 0.05, batch_size=N, replay_capacity=a.replay,
                          lockstep_envs=N, seed=7, device=local)
    L.init_params(0)
    engine.sac_train_run(env, L, (a.replay + N - 1) // N + 1, False, want_stats=False)
    engine.sac_train_run(env, L, 5, True, want_stats=False)
    torch.cuda.synchronize(dev)
    K = max(5, min(a.steps, 50))
    times = []
    t0 = time.perf_counter()
    while len(times) < 3 or time.perf_counter() - t0 < 0.5:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        engine.sac_train_run(env, L, K, True, want_stats=False)
        e1.record(stream)
        torch.cuda.synchronize(dev)
        times.append(e0.elapsed_time(e1))
    med = statistics.median(times)
    out = {"label": label, "value": N * K / (med * 1e-3), "unit": "env_steps/s", "updates_per_s": K / (med * 1e-3), "ms_per_step": med / K,
           "repeats": len(times), "n_gpus": 1,
           "config": {"workload": "%d envs, continuous update_PathPlan, SAC actor 100-64-(2,2) + 2 critics 102-64-64-2, batch %d, replay %d (> L2), "
                                  "1 update / lockstep iteration" % (N, N, a.replay)}}
    L.close(); env.close()
    return out


class PluginE2E:
    """The e2e loop: the reference-facing plug-in classes built from the XML configs the way EnvFactory / TrainerFactory
    build them, driven per step with HOST arrays at every boundary (PathPlan_City_B200.run_step_OffPolicy =
    run_thread_OffPolicy + update for all UAVs)."""

    def __init__(self, a, rank, world, local, dist):
        import importlib
        from uavrl_b200.plugins import xmlconfig
        cwd = os.getcwd()
        os.chdir(ROOT)
        try:
            cfg = xmlconfig.XML2Dict(os.path.join(ROOT, "configs", "PathPlan_City_B200.xml"))["simulator"]
            ed = cfg["env"]
            ed["num_UAV"], ed["scenario_pool"], ed["device"], ed["host_driven"], ed["seed"] = str(a.envs), str(a.pool), str(local), "1", str(42 + rank)
            ed["Agent"]["Trainer"]["Trainer_path"] = os.path.join(ROOT, "configs", "Trainer_%s_B200.xml" % {"dqn": "DQN", "ddqn": "DDQN", "dueling": "DuelingDQN"}[a.algo])
            mod = importlib.import_module("uavrl_b200.plugins." + ed["Env_Type"])
            # trainer hyper-parameters of this workload (the XML ships the reference's Batch_Size 64 / replay 10 000)
            self._patch = dict(Batch_Size=str(a.batch), replay_size=str(64 * a.envs), NetWork=NET_XML[a.net], save_loop="1000000000", model_path="/tmp/uavrl_bench_mod_%d" % os.getpid())
            orig = xmlconfig.XML2Dict

            def patched(path):
                d = orig(path)
                if "Trainer" in d and isinstance(d["Trainer"], dict):
                    d["Trainer"].update(self._patch)
                return d
            mod.XML2Dict = patched
            try:
                self.env = getattr(mod, ed["Env_Type"])(ed)
            finally:
                mod.XML2Dict = orig
        finally:
            os.chdir(cwd)
        self.tr = self.env.Trainer
        assert type(self.tr).__name__ == TRAINER_XML[a.algo]
        if world > 1:
            self.tr.attach_dist(dist, rank, world)
        N = a.envs
        ob = N * OBS * 4
        # per step: get_action (obs in, actions out) + Move_Agent (actions in; obs, reward, done, info out) + replay add (s, a, r, s2, d in) + update (loss out)
        self.h2d_bytes = ob + N * 4 + (2 * ob + N * 4 + N * 4 + N)
        self.d2h_bytes = N * 4 + (ob + N * 4 + N + N) + 4
        self.state = self.env.states()
        self.loss = 0.0

    def run(self, iters, eps):
        for _ in range(iters):
            self.state, r, d, info, res = self.env.run_step_OffPolicy(eps, self.state)
            lt = res["loss"]
            self.loss = float(lt) if not hasattr(lt, "item") else float(lt.item())      # device -> host read of the step's result
        return self.loss


def run_ours(a):
    import torch
    import torch.distributed as dist
    import uavrl_b200  # noqa: F401
    from uavrl_b200 import _lib, engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus and world > 1:
        a.gpus = world
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sampler = ClockSampler(local)
    sampler.start()                                   # every rank samples its own GPU; the fork is far from any timed region
    if world > 1:
        # NCCL prints its version banner on fd 1 at communicator creation: park stdout on stderr meanwhile so that
        # this process's stdout carries the ONE JSON line only
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier(device_ids=[local])
            torch.cuda.synchronize(dev)
        finally:
            os.dup2(saved, 1)
            os.close(saved)

    _lib.lib().uavrl_set_pdl(int(a.pdl))
    _lib.lib().uavrl_set_fuse_act_env(int(a.fuse))
    if a.fuse_dw >= 0:
        _lib.lib().uavrl_set_fuse_dw_adam(int(a.fuse_dw))
    N, B = a.envs, a.batch
    stream = torch.cuda.current_stream(dev)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize(dev)

    wl = Workload(a, rank, world, local, dist if world > 1 else None)
    env, L, tc_on = wl.env, wl.L, wl.tc_on
    wl.iterate(max(a.warmup, 3))
    torch.cuda.synchronize(dev)

    launches0 = _lib.launch_count()
    ms, t_wall, mark = timed_steps(wl, a, dev, stream, barrier, sampler)
    clocks = sampler.stop(mark)
    launches = _lib.launch_count() - launches0
    if a.dump_outputs and rank == 0:
        dump_outputs(wl, a.dump_outputs)
    value = N * world * a.steps / (ms * 1e-3)
    if world > 1:       # every rank's clock record, gathered
        allc = [None] * world
        dist.all_gather_object(allc, clocks)
        clocks = dict(allc[0], per_rank=[{k: c.get(k) for k in ("sm_mhz", "sm_min_mhz", "reasons", "samples")} for c in allc])

    out = None
    if rank == 0:
        pk = measured_peaks()
        out = {"metric": "env steps/sec (+ DQN updates/sec), 500x500x100 city", "value": value, "unit": "env_steps/s",
               "updates_per_s": a.steps / (ms * 1e-3), "samples_per_s": a.steps * B * world / (ms * 1e-3),
               "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms / a.steps,
               "timed_ms": ms, "timed_region_s": t_wall,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "f64 env state / f32 obs+learner", "data": "synthetic",
               "config": dict(config_dict(a, world), qnet_path=("tcgen05 3xTF32 (fp32-grade)" if tc_on else "fp32 CUDA cores"),
                              launch=("programmatic dependent launch" if a.pdl else "serialised")
                              + (", get_action+step fused" if (a.fuse and tc_on) else ""),
                              timing="the %d timed steps as one block (barrier + synchronize both sides, CUDA events, max over ranks)"
                                     % a.steps),
               "clocks": clocks, "gpu_launches": int(launches),
               "host_wall_ms_per_step": 1e3 * t_wall / a.steps}

    # ---- roofline pass: per-kernel CUDA-event time (rank 0's GPU; same workload, events between kernels)
    if rank == 0:
        n_prof = max(50, min(a.steps, 200))
        kp = engine.train_profile(env, L, n_prof, a.eps) / float(n_prof)   # ms per launch
        fused = bool(a.fuse) and tc_on
        names = ("act+env_step_fused" if fused else "act_eps_greedy", "env_step", "td_target", "fwd_bwd", "weight_grad", "reduce_adam")
        fwd = FWD_FLOPS[a.net]
        n_tgt = 1 if a.algo == "dqn" else 2          # target fwd (+ local fwd on s' for double DQN)
        # SURVEY 8(d): per sampled transition 4x fwd (DQN) / 5x fwd (DDQN) = target pass(es) + fwd on s + backward (2 fwd)
        if tc_on:
            alg_flops = {"act_eps_greedy": fwd * N, "env_step": 0, "td_target": n_tgt * fwd * B, "fwd_bwd": 2 * fwd * B,
                         "weight_grad": fwd * B, "reduce_adam": 0}
            alg_bytes = {"act_eps_greedy": ACT_BYTES * N, "env_step": ENV_STEP_BYTES * N, "td_target": (OBS * 4 + 9) * B * n_tgt,
                         "fwd_bwd": (OBS * 4 + 8) * B, "weight_grad": OBS * 4 * B, "reduce_adam": 28 * L.P}
        else:
            alg_flops = {"act_eps_greedy": fwd * N, "env_step": 0, "td_target": 0, "fwd_bwd": (n_tgt + 3) * fwd * B,
                         "weight_grad": 0, "reduce_adam": 0}
            alg_bytes = {"act_eps_greedy": ACT_BYTES * N, "env_step": ENV_STEP_BYTES * N, "td_target": 0,
                         "fwd_bwd": TRANSITION_BYTES * B, "weight_grad": 0, "reduce_adam": 28 * L.P}
        if fused:
            for dct in (alg_flops, alg_bytes):
                dct["act+env_step_fused"] = dct["act_eps_greedy"] + dct["env_step"]
        td_fused = tc_on and L.td_fused(B)
        if td_fused:
            # the TD-target pass(es) run inside the training kernel (uavrl_set_fuse_td): one launch carries both rows' work;
            # the profile's td_target slot then brackets no launch at all (event overhead only) and is dropped
            names = tuple("td_target+fwd_bwd" if n_ == "fwd_bwd" else n_ for n_ in names)
            for dct in (alg_flops, alg_bytes):
                dct["td_target+fwd_bwd"] = dct["td_target"] + dct["fwd_bwd"]
        kernels = {}
        for n_, t_ in zip(names, kp):
            if t_ <= 0 or (td_fused and n_ == "td_target"):
                continue
            kernels[n_] = {"ms": float(t_), "share": float(t_ / kp.sum()), "GBps": alg_bytes[n_] / (t_ * 1e-3) / 1e9,
                           "TFLOPs": alg_flops[n_] / (t_ * 1e-3) / 1e12}
        dom = max(kernels, key=lambda k: kernels[k]["ms"])
        if alg_flops[dom] > 0:
            ach = kernels[dom]["TFLOPs"]
            roof = {"kernel": dom, "bound": "tensor", "achieved": ach, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                    "frac": ach / pk["tf_sustained"], "traffic": None,
                    "note": ("3xTF32 tcgen05 path: 3 tensor-core products per algorithmic product, " if tc_on else "fp32 CUDA-core path, ")
                            + "measured against the %s bf16 tensor peak; HBM view %.1f GB/s of %.0f"
                            % (pk["src"], kernels[dom]["GBps"], pk["hbm"])}
        else:
            ach = kernels[dom]["GBps"]
            roof = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s",
                    "frac": ach / pk["hbm"], "traffic": None}
        # dram bytes per launch of the same kernel from the committed `ncu --set full` capture of this exact command
        # (profiles/r02_ncu_traffic.json; only valid for the workload it was captured on, replay size included)
        try:
            with open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")) as f:
                tr = json.load(f)
            same = (tr.get("envs") == N and tr.get("batch") == B and tr.get("net") == a.net and tr.get("algo") == a.algo
                    and bool(tr.get("tc")) == bool(tc_on) and tr.get("replay") == a.replay)
            if same:
                roof["traffic"] = tr["dram_bytes_per_launch"].get(dom)
                roof["traffic_source"] = tr.get("source")
        except (OSError, ValueError, KeyError):
            pass
        roof["peak_source"] = pk["src"]
        roof["algorithmic_bytes_per_launch"] = alg_bytes[dom]
        out["roofline"] = roof
        out["kernels"] = kernels
        # the whole iteration against HBM: algorithmic bytes of all six kernels / the timed iteration
        tot_bytes = sum(alg_bytes[k] for k in kernels)
        out["iteration_hbm"] = {"algorithmic_bytes": tot_bytes, "GBps": tot_bytes / (ms / a.steps * 1e-3) / 1e9,
                                "frac_of_hbm_peak": tot_bytes / (ms / a.steps * 1e-3) / 1e9 / pk["hbm"]}

    # ---- e2e: the same iteration through the plug-in classes, host arrays at every boundary
    if not a.no_e2e:
        pe = PluginE2E(a, rank, world, local, dist if world > 1 else None)
        pe.run(5, a.eps)                     # fills the replay past Batch_Size, warms the pinned rings
        barrier()
        ke = max(20, min(a.steps, 100))
        blocks = []
        t_all = time.perf_counter()
        while len(blocks) < 3 or time.perf_counter() - t_all < 0.5:
            barrier()
            t0 = time.perf_counter()
            pe.run(ke, a.eps)
            torch.cuda.synchronize(dev)
            dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            blocks.append(float(dt.item()))
            if world > 1:       # same number of blocks on every rank
                go = torch.tensor([1.0 if (len(blocks) < 3 or time.perf_counter() - t_all < 0.5) else 0.0], device=dev)
                dist.broadcast(go, 0)
                if go.item() == 0.0:
                    break
        dt = statistics.median(blocks)
        if rank == 0:
            out["e2e"] = {"value": N * world * ke / dt, "unit": "env_steps/s", "h2d_bytes_per_step": pe.h2d_bytes,
                          "d2h_bytes_per_step": pe.d2h_bytes, "steps": ke, "repeats": len(blocks), "ms_per_step": 1e3 * dt / ke,
                          "what": "per step through PathPlan_City_B200.run_step_OffPolicy + %s (plug-in classes built from configs/*.xml): "
                                  "get_action(host obs)->host actions, Move_Agent(host actions)->host obs/reward/done/info, replay add from host "
                                  "arrays, update()->host loss; pinned host memory, copies inside the timed region%s"
                                  % (TRAINER_XML[a.algo], "; gradient exchange = the fused NVLink all-reduce + Adam" if world > 1 else "")}

    # ---- the other BASELINE configs that fit this launch
    if not a.no_configs:
        subs = {}
        if world == 1:
            # a fixed count of its own: about 0.5 s at the 0.1 ms per step this config takes on one B200
            a2 = argparse.Namespace(**vars(a)); a2.envs = a2.batch = 16384; a2.net, a2.algo = "vanet2", "dueling"; a2.steps = 5000
            subs["configs[2]"] = measure_config(a2, rank, world, local, None, dev, stream, barrier,
                                                "16384 envs, DuelingDQN (VAnet2), buildings.xml obstacle set, 1xB200")
            subs["configs[4]"] = measure_sac(a, local, dev, stream, "16384 envs, SAC_Trainer continuous-action UAV (actor+2 critics), 1xB200")
        if world == 8:
            # about 0.5 s: this per-GPU shape takes 73 us per step on one B200, plus the gradient exchange
            a3 = argparse.Namespace(**vars(a)); a3.envs = a3.batch = 8192; a3.net, a3.algo = "qvalue3", "ddqn"; a3.steps = 6000
            subs["configs[3]"] = measure_config(a3, rank, world, local, dist, dev, stream, barrier,
                                                "65536 envs (8192/GPU), DDQN, replay buffer 1M/GPU, grad allreduce across 8xB200")
        if rank == 0 and subs:
            out["configs"] = subs

    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(a, a.cpu_seconds)
    if rank == 0:
        print(json.dumps(out, default=float), flush=True)
    sys.stdout.flush()
    if world > 1:
        dist.barrier(device_ids=[local])
    wl.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.steps is None:
        args.steps = 200 if args.impl == "reference" else 25000
    if args.batch <= 0:
        args.batch = args.envs
    usable_cpus()                           # read the affinity mask before any OpenMP runtime can pin this thread
    cpu_env(args.threads, bind=(args.impl == "reference"))
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)
