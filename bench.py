#!/usr/bin/env python
"""Rollout benchmark: env-steps/s of the PPO rollout phase (policy act + crowd_sim step +
rollout-storage insert, auto-resets included) on BASELINE.json config[1]:
CrowdSimPred-v0 / const_vel / 20 humans / HH+HR attention / 4096 environments per B200.

    python bench.py --gpus N --steps K --warmup W          # ours (torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU arm: the unmodified reference on the host cores

One "step" = one rollout step of every environment of the job.  Prints ONE JSON line (rank 0).
  value    : device-resident rollout (inputs already in HBM, no host round trip), CUDA-event timed
  e2e      : the same loop through the reference-facing VecEnv/Policy API — reward/done/info come
             back to the host every step and masks/rewards go host->device into the storage,
             exactly what the unchanged train.py loop does (train.py:177-191)
  roofline : the dominant kernel of the step, picked from the live per-kernel timing (the environment step kernel:
             algorithmic bytes / CUDA-event time vs the measured HBM copy bandwidth); `roofline_other` = the largest
             tensor-core launch (QKV projection GEMM: algorithmic FLOPs vs the measured sustained bf16 peak)
  update   : one PPO update (5 epochs x 2 minibatches) on the rollout just collected, gradient all-reduce over NCCL
             active when n_gpus > 1 (time and share from CUDA events around the collective)
  configs  : BASELINE configs[2..4] (c3 GST wrapper, c4 50 randomised humans, c5 100 humans) -- same device-resident
             rollout step and one PPO update each, at the run's world size
  cpu_baseline : the UNMODIFIED reference rollout (ShmemVecEnv fork workers + reference Policy on CPU, behind
             oracle/shims) when tools/stage_reference.py has staged it under baseline/_ref (kind "reference"),
             else the oracle port (kind "port"); bounded sample, host cores stated
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

METRIC = "env_steps_per_s_ppo_rollout"
UNIT = "env-steps/s"
HUMANS = 20
ENVS_PER_GPU = 4096
ROLLOUT_T = 30
B_ENV = 4 * (23 * HUMANS + 22) + 4 * (2 * 6 * HUMANS + 11) + 2      # SURVEY.md §8d: 2934 B
B_POL = 4 * (2 * 6 * HUMANS + 10) + 1044                              # 2044 B


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=90)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--gemm-mode", type=int, default=int(os.environ.get("CN_GEMM_MODE", "1")),
                    help="1 = tcgen05 3xFP16 GEMMs (default), 0 = fp32 CUDA-core GEMMs")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-update", action="store_true", help="skip the PPO update blocks (rollout numbers only)")
    ap.add_argument("--configs", default="c3,c4,c5", help="other BASELINE configs reported in the `configs` block ('' = none)")
    ap.add_argument("--config-steps", type=int, default=60)
    ap.add_argument("--config-burn-in", type=int, default=150)
    ap.add_argument("--burn-in", type=int, default=400,
                    help="untimed rollout steps before the warm-up: all environments start their first episode "
                         "in lock-step (a transient with ~25 %% more work per step, tools/step_series.py); a "
                         "training run lives in the desynchronised steady state reached after ~250 steps")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (rank 0) as DIR/<name>.npy "
                         "(float32); the same arguments give the same inputs, so two builds can be compared")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------ CPU arm
def _cpu_worker(args):
    """One host process: k oracle environments + the PyTorch fp32 oracle policy, W + K rollout steps."""
    widx, k, warmup, steps, seed = args
    import numpy as np
    import torch
    torch.set_num_threads(1)
    try:                       # numpy's BLAS pool must not oversubscribe the cores (one worker per core)
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:
        pass
    from oracle.crowd_env import EnvConfig, OracleVecEnv
    from oracle.policy_ref import PolicyRef
    env = OracleVecEnv(EnvConfig(human_num=HUMANS), k, seed=seed, rank_offset=widx * k, nenv_total=1 << 20)
    torch.manual_seed(425)
    pol = PolicyRef(12)
    obs = env.reset()
    h = torch.zeros(k, 1, 128)
    masks = torch.ones(k, 1)
    std = pol.logstd().exp().detach()
    t0 = None
    for s in range(warmup + steps):
        if s == warmup:
            t0 = time.perf_counter()
        with torch.no_grad():
            value, mean, h = pol({kk: torch.from_numpy(v) for kk, v in obs.items()}, h, masks)
            action = mean + std * torch.randn_like(mean)
        obs, rew, done, infos = env.step(action.numpy())
        masks = torch.from_numpy(1.0 - done.astype(np.float32)).reshape(k, 1)
    return time.perf_counter() - t0


def cpu_rollout_rate(steps, warmup, envs_per_worker=4, workers=None):
    """env-steps/s of the oracle port using every host core (fork workers, like ShmemVecEnv)."""
    import multiprocessing as mp
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[v] = "1"
    workers = workers or len(os.sched_getaffinity(0)) or (os.cpu_count() or 1)
    ctx = mp.get_context("fork")
    with ctx.Pool(workers) as pool:
        times = pool.map(_cpu_worker, [(w, envs_per_worker, warmup, steps, 425) for w in range(workers)])
    total = workers * envs_per_worker * steps
    ts = sorted(times)
    return total / max(times), workers, envs_per_worker, (ts[len(ts) // 2], ts[-1])


def _reference_root():
    """Unmodified reference staged by tools/stage_reference.py (travels to the GPU box), else the checkout."""
    for p in (os.path.join(REPO, "baseline", "_ref"), "/root/reference"):
        if os.path.isfile(os.path.join(p, "rl", "networks", "shmem_vec_env.py")):
            return p
    return None


def reference_rollout_rate(steps, warmup, num_processes=None, humans=HUMANS):
    """env-steps/s of the UNMODIFIED reference rollout on the host cores (SURVEY.md §8d 'CPU baseline timing'):
    rl.networks.envs.make_vec_envs -> ShmemVecEnv with one fork worker per environment (the reference's own
    design: one OS process per env), reference Policy.act on CPU in the parent with all host threads, config 2
    (CrowdSimPred-v0 / const_vel / 20 humans, fixed attributes), behind oracle/shims for the un-vendored
    gym / baselines / rvo2.  Returns a dict (rate + per-step timing spread), or None if no reference is staged."""
    root = _reference_root()
    if root is None:
        return None
    subprocess.check_call(["make", "-s", "-C", os.path.join(REPO, "oracle")])
    sys.path[:0] = [os.path.join(REPO, "oracle", "shims"), root]
    cores = len(os.sched_getaffinity(0)) or (os.cpu_count() or 1)
    n = num_processes or cores
    # The fork workers must be single-threaded: they inherit the parent's OpenMP / BLAS pools, and on a 128-core box
    # 128 workers x 128 spinning threads each never finish a step (the first version of this arm timed out after 600 s
    # there).  So the pools are limited to 1 thread BEFORE the workers are forked and only the parent's torch pool is
    # widened afterwards (the policy forward and the env steps alternate, they never compete for the cores).
    pol_threads = min(cores, 32)
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[v] = "1"
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:
        pass
    verbose = os.environ.get("CN_BENCH_VERBOSE", "0") == "1"
    t_start = time.perf_counter()

    def note(msg):
        if verbose:
            sys.stderr.write("[reference arm %.1fs] %s\n" % (time.perf_counter() - t_start, msg))
            sys.stderr.flush()
    argv, sys.argv = sys.argv, ["x", "--no-cuda", "--env-name", "CrowdSimPred-v0", "--num-processes", str(n)]
    cwd = os.getcwd()
    os.chdir(root)
    try:
        import numpy as np
        import torch
        import rvo2
        torch.set_num_threads(1)
        rvo2.ONLY_AGENT0 = False                     # the reference's full doStep (H agents per cached simulator)
        from arguments import get_args
        from crowd_nav.configs.config import Config
        from rl.networks.envs import make_vec_envs
        from rl.networks.model import Policy
        import crowd_sim  # noqa: F401  (registers the gym ids)
        args = get_args()
        config = Config()
        # BASELINE config 2 through the reference's own Config object (what a user sets in config.py)
        config.sim.predict_method, config.env.use_wrapper = 'const_vel', False
        config.sim.human_num = humans
        config.env.randomize_attributes, config.humans.random_goal_changing = False, False
        import io, contextlib
        with contextlib.redirect_stdout(io.StringIO()):          # make_env prints one Monitor repr per environment
            envs = make_vec_envs("CrowdSimPred-v0", 425, n, args.gamma, None, torch.device("cpu"), False, config=config,
                                 pretext_wrapper=False)
        note("make_vec_envs done (%d workers)" % n)
        torch.manual_seed(425)
        torch.set_num_threads(pol_threads)
        pol = Policy(envs.observation_space.spaces, envs.action_space, base_kwargs=args, base='selfAttn_merge_srnn')
        obs = envs.reset()
        note("reset done")
        hx = {'human_node_rnn': torch.zeros(n, 1, 128), 'human_human_edge_rnn': torch.zeros(n, humans + 1, 256)}
        masks = torch.ones(n, 1)
        t_env, t_pol = [], []
        for s in range(warmup + steps):
            t0 = time.perf_counter()
            with torch.no_grad():
                value, action, logp, hx = pol.act(obs, hx, masks)
            t1 = time.perf_counter()
            obs, rew, done, infos = envs.step(action)
            masks = torch.FloatTensor([[0.0] if d else [1.0] for d in done])
            t2 = time.perf_counter()
            if s >= warmup:
                t_pol.append(t1 - t0)
                t_env.append(t2 - t1)
            if s < 3 or s % 50 == 0:
                note("step %d: policy %.1f ms, env %.1f ms" % (s, 1e3 * (t1 - t0), 1e3 * (t2 - t1)))
        envs.close()
    finally:
        os.chdir(cwd)
        sys.argv = argv
    tot = sum(t_env) + sum(t_pol)
    return dict(rate=n * steps / tot, workers=n, cores=cores, steps=steps, pol_threads=pol_threads,
                env_ms_median=1e3 * float(np.median(t_env)), env_ms_max=1e3 * float(np.max(t_env)),
                policy_ms_median=1e3 * float(np.median(t_pol)), policy_ms_max=1e3 * float(np.max(t_pol)),
                env_only_rate=n * steps / sum(t_env), root=os.path.relpath(root, REPO) if root.startswith(REPO) else root)


def cpu_arm(steps, warmup, seconds=None):
    """The CPU arm both bench legs report: the unmodified reference when it is staged (kind 'reference'),
    else the oracle port (kind 'port').  Returns (rate, cpu_baseline dict)."""
    if _reference_root() is not None:
        if seconds is not None:          # bounded sample: ~25 ms per env-step per core => steps for `seconds` of wall time
            steps = max(4, int(seconds / 0.06))
        r = reference_rollout_rate(steps, warmup)
        sample = ("UNMODIFIED reference (%s): make_vec_envs -> ShmemVecEnv, %d fork workers x 1 env (one process per env, "
                  "the reference's design), reference Policy.act on CPU (%d torch threads), CrowdSimPred-v0 const_vel H=%d, "
                  "%d rollout steps after %d warm-up; per step: env %.1f ms median / %.1f ms max, policy %.1f ms median / "
                  "%.1f ms max; env-only %.0f env-steps/s; behind oracle/shims (gym, baselines, rvo2 = oracle/rvo2_ref.cpp)"
                  % (r["root"], r["workers"], r["pol_threads"], HUMANS, r["steps"], warmup, r["env_ms_median"], r["env_ms_max"],
                     r["policy_ms_median"], r["policy_ms_max"], r["env_only_rate"]))
        return r["rate"], {"value": r["rate"], "unit": UNIT, "cores": r["cores"], "kind": "reference", "sample": sample,
                           "workers": r["workers"], "detail": {k: r[k] for k in (
                               "env_ms_median", "env_ms_max", "policy_ms_median", "policy_ms_max", "env_only_rate")}}
    if seconds is not None:
        steps = max(4, int(seconds / 0.035))
    rate, workers, k, spread = cpu_rollout_rate(steps, warmup)
    sample = ("oracle PORT (no staged reference): %d fork workers x %d oracle envs x %d rollout steps (oracle/crowd_env.py + "
              "rvo2_ref.cpp + policy_ref.py, torch fp32, 1 thread each); worker seconds median %.2f / max %.2f"
              % (workers, k, steps, spread[0], spread[1]))
    return rate, {"value": rate, "unit": UNIT, "cores": workers, "kind": "port", "sample": sample}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.perf_counter()
    rate, base = cpu_arm(a.steps, a.warmup)
    wall = time.perf_counter() - t0
    envs = base.get("workers", base["cores"])
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1000.0 * envs / rate, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "CrowdSimPred-v0 const_vel, 20 humans, HH+HR attention rollout (bounded CPU sample: %d envs)" % envs,
                   "parallelism": "%d host processes" % envs},
        "cpu_baseline": base,
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": wall,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ GPU arm
class ClockSampler(object):
    def __init__(self, index):
        self.path = tempfile.mktemp(suffix=".csv")
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = []
        for ln in open(self.path).read().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) >= 7 and f[0].replace(".", "").isdigit():
                rows.append(f)
        os.unlink(self.path)
        if not rows:
            return out
        sm = sorted(float(r[0]) for r in rows)
        hot = [x for x in sm if x >= 0.5 * max(sm)] or sm
        out["sm_mhz"] = hot[len(hot) // 2]
        out["sm_max_mhz"] = float(rows[0][1])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        out["reasons"] = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows)]
        out["samples"] = len(rows)
        try:
            out["power_w_max"] = max(float(r[2]) for r in rows)
        except ValueError:
            pass
        return out


def _bind_numa(local, nlocal):
    """Pin this rank to the host cores next to its GPU (or an even share of the cores when the topology cannot be
    read): with 8 unpinned ranks the reference-facing loop's host work (one ctypes call, one D2H + sync and a few numpy
    copies per step) migrated between sockets and the 8-GPU e2e efficiency fell to 0.69 in round 1."""
    try:
        import torch
        cores = sorted(os.sched_getaffinity(0))
        node_cpus = None
        bus = torch.cuda.get_device_properties(local).pci_bus_id if hasattr(torch.cuda.get_device_properties(local), "pci_bus_id") else None
        if bus is not None:
            dom = torch.cuda.get_device_properties(local).pci_domain_id
            devid = torch.cuda.get_device_properties(local).pci_device_id
            path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, devid)
            if os.path.exists(path):
                node = int(open(path).read().strip())
                cl = "/sys/devices/system/node/node%d/cpulist" % node
                if node >= 0 and os.path.exists(cl):
                    cpus = []
                    for part in open(cl).read().strip().split(","):
                        lo, _, hi = part.partition("-")
                        cpus.extend(range(int(lo), int(hi or lo) + 1))
                    node_cpus = [c for c in cpus if c in cores]
        if node_cpus and len(node_cpus) >= 4:
            share = node_cpus          # all ranks of this node share its cores (the loop is one thread + torch helpers)
            how = "numa node of the GPU (%d cores)" % len(share)
        else:
            per = max(1, len(cores) // max(1, nlocal))
            share = cores[local * per:(local + 1) * per] or cores
            how = "even split (%d cores)" % len(share)
        os.sched_setaffinity(0, share)
        return how
    except Exception as e:          # affinity is an optimisation, never a failure
        return "unbound (%s)" % (repr(e)[:80],)


EXTRA_CONFIGS = {
    # BASELINE configs[2]: CrowdSimPredRealGST-v0 + GST predictor wrapper, 20 humans, 4096 envs per GPU
    "c3": dict(kind="gst", H=20, envs=4096, kw=dict(human_num=20),
               workload="CrowdSimPredRealGST-v0 inferred GST predictor, 20 humans (BASELINE configs[2])"),
    # BASELINE configs[3]: CrowdSimPred-v0 randomised ORCA, 50 humans, 16384 envs over 8 GPUs = 2048 per GPU
    "c4": dict(kind="pred", H=50, envs=2048, kw=dict(human_num=50, randomize_attributes=1, random_goal_changing=1,
                                                     goal_change_chance=0.5),
               workload="CrowdSimPred-v0 randomised ORCA (attributes + goal changes), 50 humans (BASELINE configs[3])"),
    # BASELINE configs[4]: dense 100-human crowd, 32768 envs over 8 GPUs = 4096 per GPU.  The reference cannot place
    # more than ~76 humans on its 6*sqrt(2) m circle (generate_circle_crossing_human loops forever,
    # crowd_sim_var_num.py:118-141), so the circle and the arena are scaled by 2 here; spawn_overflow_envs counts the
    # environments where a rejection-sampling loop still hit the 20 000-try cap.
    # num_mini_batch 8 for the update (train.py's default 2 would need > 40 GB per padded attention tensor at H = 100).
    "c5": dict(kind="pred", H=100, envs=4096, mini_batches=8,
               kw=dict(human_num=100, circle_radius=2 * 6 * 2 ** 0.5, arena_size=12.0),
               workload="dense 100-human crowd, HH+HR attention, sim.circle_radius and arena_size x2 so that the reference's "
                        "spawner can place 100 humans (BASELINE configs[4])"),
}


def _ppo_update_block(torch, policy, rollouts, world, envs, mini_batches=2):
    """One PPO update (5 epochs x 2 minibatches, train.py defaults) on the rollout just collected, with the NCCL gradient
    all-reduce active when world > 1.  Device-timed; the all-reduce share comes from CUDA events around the collective."""
    from crowdnav_prediction_attngraph_b200 import ppo
    agent = ppo.PPO(policy, 0.2, 5, mini_batches, 0.5, 0.0, lr=4e-5, eps=1e-5, max_grad_norm=0.5)
    agent.profile = True
    with torch.no_grad():
        o = {k: rollouts.obs[k][-1] for k in rollouts.obs}
        hx = {'human_node_rnn': rollouts.recurrent_hidden_states['human_node_rnn'][-1]}
        nv = policy.get_value(o, hx, rollouts.masks[-1]).detach()
    rollouts.compute_returns(nv, True, 0.99, 0.95, False)
    try:
        # one untimed update first: the first call pays one-time costs (caching-allocator growth to ~10 GB, cuBLAS /
        # kernel-attribute initialisation: 1.2-1.8 s), a training run pays them once in thousands of updates
        agent.update(rollouts)
        torch.cuda.synchronize()
        # two timed updates, the faster one is reported: the compacted row counts differ from minibatch to minibatch, so
        # the caching allocator can still grow (cudaMalloc + implicit sync) in the update right after the warm-up one
        samples, prof = [], {}
        for _ in range(2):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            agent.update(rollouts)
            e1.record()
            torch.cuda.synchronize()
            samples.append(e0.elapsed_time(e1))
            if samples[-1] == min(samples):
                prof = agent.last_profile or {}
    except torch.cuda.OutOfMemoryError as e:
        torch.cuda.empty_cache()
        return {"ms": 0.0, "error": "out of memory: " + str(e)[:160], "num_mini_batch": mini_batches}
    rollouts.after_update()
    ms = min(samples)
    return {"ms": ms, "samples": envs * ROLLOUT_T, "ppo_epoch": 5, "num_mini_batch": mini_batches,
            "optimizer_steps": 5 * mini_batches,
            "allreduce_ms": prof.get("allreduce_ms", 0.0), "allreduce_calls": prof.get("allreduce_calls", 0),
            "allreduce_bytes_per_call": prof.get("allreduce_bytes_per_call", 0),
            "allreduce_share": (prof.get("allreduce_ms", 0.0) / ms) if ms > 0 else None,
            "collective": "NCCL all-reduce of the flat fp32 gradient before clip_grad_norm_ (rl/ppo/ppo.py:83-86), world %d" % world,
            "kernels": "tcgen05 3xFP16 linear layers (fwd / dgrad / split-K wgrad), compacted-row attention fwd/bwd, fused GRU "
                       "sequence (CN_UPDATE_KERNELS=1)" if os.environ.get("CN_UPDATE_KERNELS", "1") == "1" else "plain torch ops",
            "ms_samples": samples,
            "timing": "faster of two timed updates on the same rollout, after one untimed update that pays allocator / library warm-up",
            "peak_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}


def _run_extra_config(torch, dist, name, spec, dev, rank, world, steps, warmup, burn_in, with_update):
    """Device-resident rollout (same zero-copy step as the headline `value`) of another BASELINE config, then one PPO
    update with the gradient all-reduce.  Returns the per-rank dict; the caller reduces the times over ranks."""
    import numpy as np
    from crowdnav_prediction_attngraph_b200.vec_env import CudaCrowdVecEnv, CudaPretextVecEnv
    from crowdnav_prediction_attngraph_b200.policy import Policy
    from crowdnav_prediction_attngraph_b200.storage import RolloutStorage
    N, H = spec["envs"], spec["H"]
    common = dict(num_envs=N, nenv_total=N * world, rank_offset=rank * N, seed=425, device=dev)
    if spec["kind"] == "gst":
        params = dict(np.load(os.path.join(REPO, "tests", "golden", "gst_params.npz")))
        env = CudaPretextVecEnv(params, **common, **spec["kw"])
    else:
        env = CudaCrowdVecEnv(**common, **spec["kw"])

    class Args(object):
        num_processes, seq_length, num_mini_batch = N, ROLLOUT_T, 2
    torch.manual_seed(425)
    policy = Policy(env.observation_space.spaces, env.action_space, base_kwargs=Args(), base='selfAttn_merge_srnn').to(dev)
    rollouts = RolloutStorage(ROLLOUT_T, N, env.observation_space.spaces, env.action_space, 128, 256, device=dev)
    obs = env.reset()
    for k in rollouts.obs:
        rollouts.obs[k][0].copy_(obs[k])
    eng = policy._engine(N, dev)

    if spec["kind"] == "gst":
        # the wrapper's kernel produces the observation in its own buffers: act -> step -> fused insert (one launch)
        def device_step():
            s = rollouts.step
            o = {k: rollouts.obs[k][s] for k in rollouts.obs}
            hn = rollouts.recurrent_hidden_states['human_node_rnn']
            eng.act(o, hn[s], rollouts.masks[s], out=dict(value=rollouts.value_preds[s], action=rollouts.actions[s],
                                                          log_prob=rollouts.action_log_probs[s], h_out=hn[s + 1]))
            nobs, rew, done, info = env.step_device(rollouts.actions[s])
            rollouts.insert(nobs, {'human_node_rnn': hn[s + 1]}, rollouts.actions[s], rollouts.action_log_probs[s],
                            rollouts.value_preds[s], rew, (1.0 - done.float()).unsqueeze(1))
            if rollouts.step == 0:
                rollouts.after_update()
    else:
        def device_step():
            rollouts.rollout_step_zero_copy(eng, env)
            if rollouts.step == 0:
                rollouts.after_update()
    for _ in range(burn_in + warmup):
        device_step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    while rollouts.step != 0:                     # start the timed region on a rollout boundary
        device_step()
    l0 = env.launch_count() + eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        device_step()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    out = {"ms_total": ms, "launches": env.launch_count() + eng.launch_count() - l0,
           "valid_human_rows": int(eng.lib.cn_policy_last_rows(eng._h)),
           "spawn_overflow_envs": int(env.get_state("spawn_overflow").sum()),
           "deferred_events": int(env.get_state("defer_ctl")[2])}
    if with_update:
        while rollouts.step != 0:
            device_step()
        out["update"] = _ppo_update_block(torch, policy, rollouts, world, N, spec.get("mini_batches", 2))
    env.close()
    del eng, policy, rollouts, env
    torch.cuda.empty_cache()
    return out


DUMP_MAX_BYTES = 64 << 20


def dump_last_step(rollouts, out_dir):
    """Write what the last device_step returned to its caller: the policy's value / action / log-prob / hidden state
    and the environment's next observation / reward / not-done mask, from the storage slot that step filled.  Above
    DUMP_MAX_BYTES a fixed seeded sample of environments is written, their indices in env_index.npy."""
    import numpy as np
    import torch
    s = (rollouts.step - 1) % rollouts.num_steps
    out = {"value": rollouts.value_preds[s], "action": rollouts.actions[s], "action_log_prob": rollouts.action_log_probs[s],
           "hidden_state": rollouts.recurrent_hidden_states['human_node_rnn'][s + 1], "reward": rollouts.rewards[s],
           "not_done": rollouts.masks[s + 1]}
    out.update({"obs_" + k: v[s + 1] for k, v in rollouts.obs.items()})
    n = rollouts.rewards.size(1)
    per_env = sum(4 * v[0].numel() for v in out.values())
    if per_env * n > DUMP_MAX_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_BYTES // (per_env + 4), replace=False))
        idx = torch.from_numpy(keep).to(rollouts.rewards.device)
        out = {k: v.index_select(0, idx) for k, v in out.items()}
        out["env_index"] = idx
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v.float().cpu().numpy())


def run_ours(a):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    affinity = _bind_numa(local, int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))) if world > 1 else "single rank: unbound"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    from crowdnav_prediction_attngraph_b200 import _capi
    if not os.path.exists(_capi.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    from crowdnav_prediction_attngraph_b200.vec_env import CudaCrowdVecEnv, Box
    from crowdnav_prediction_attngraph_b200.policy import Policy
    from crowdnav_prediction_attngraph_b200.storage import RolloutStorage

    N = a.envs_per_gpu
    env = CudaCrowdVecEnv(num_envs=N, nenv_total=N * world, rank_offset=rank * N, seed=425, human_num=HUMANS, device=dev)

    class Args(object):
        num_processes, seq_length, num_mini_batch = N, ROLLOUT_T, 2
    torch.manual_seed(425)
    policy = Policy(env.observation_space.spaces, env.action_space, base_kwargs=Args(), base='selfAttn_merge_srnn').to(dev)
    policy._cuda = None
    os.environ["CN_GEMM_MODE"] = str(a.gemm_mode)
    rollouts = RolloutStorage(ROLLOUT_T, N, env.observation_space.spaces, env.action_space, 128, 256, device=dev)
    obs = env.reset()
    for k in rollouts.obs:
        rollouts.obs[k][0].copy_(obs[k])
    eng = policy._engine(N, dev)
    launches0 = env.launch_count() + eng.launch_count()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------------------------------------------------------- device-resident rollout (value)
    def device_step():
        rollouts.rollout_step_zero_copy(eng, env)
        if rollouts.step == 0:
            rollouts.after_update()

    for _ in range(a.burn_in):
        device_step()
    for _ in range(a.warmup):
        device_step()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    l0 = env.launch_count() + eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    c0 = time.perf_counter()
    for _ in range(a.steps):
        device_step()
    cpu_enqueue_ms = (time.perf_counter() - c0) * 1000.0 / a.steps      # host time to enqueue one step
    e1.record()
    barrier()
    ms_value = e0.elapsed_time(e1)
    launches = env.launch_count() + eng.launch_count() - l0
    if a.dump_outputs and rank == 0:
        dump_last_step(rollouts, a.dump_outputs)

    # ---------------------------------------------------------------- e2e: reference-facing API, host round trips
    # pinned staging for the host tensors train.py builds every step (masks / bad_masks / reward): allocated ONCE
    # (round 1 called .pin_memory() = cudaHostAlloc three times per step, which serialises across the 8 ranks)
    pin_masks, pin_bad, pin_rew = (torch.zeros(N, 1).pin_memory(), torch.ones(N, 1).pin_memory(), torch.zeros(N, 1).pin_memory())

    def e2e_step():
        s = rollouts.step
        o = {k: rollouts.obs[k][s] for k in rollouts.obs}
        hx = {'human_node_rnn': rollouts.recurrent_hidden_states['human_node_rnn'][s]}
        with torch.no_grad():
            value, action, logp, hx2 = policy.act(o, hx, rollouts.masks[s])
        nobs, reward, done, infos = env.step(action)          # reward CPU tensor, done numpy, lazy infos (D2H + sync inside)
        # the stream is idle after env.step's synchronize, so the staging buffers of the previous step are free again
        pin_masks.copy_(torch.from_numpy(1.0 - done.astype("float32")).unsqueeze(1))
        pin_rew.copy_(reward)
        rollouts.insert(nobs, hx2, action, logp, value, pin_rew, pin_masks, pin_bad)   # H2D copies inside
        if rollouts.step == 0:
            rollouts.after_update()
        return done

    for _ in range(max(3, a.warmup // 2)):
        e2e_step()
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    f0.record()
    for _ in range(a.steps):
        e2e_step()
    f1.record()
    barrier()
    wall_e2e = (time.perf_counter() - w0) * 1000.0
    ms_e2e = max(f0.elapsed_time(f1), 0.0)
    # the timed regions last tens of milliseconds, shorter than nvidia-smi's sampling period: keep the
    # SAME device step running (untimed) until the sampler has seen >= 1 s of load, then read it
    t_load = time.perf_counter()
    while time.perf_counter() - t_load < 1.2:
        for _ in range(50):
            device_step()
        torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    if clocks is not None:
        clocks["window"] = "warm-up + timed regions + 1.2 s of the same device step (sampling period 50 ms)"

    # ---------------------------------------------------------------- per-kernel timing (outside the timed regions)
    lib = eng.lib
    lib.cn_policy_profile(eng._h, 1)
    ns = lib.cn_policy_stage_count()
    import ctypes as C
    names = [lib.cn_policy_stage_name(i).decode() for i in range(ns)]
    acc = [0.0] * ns
    env_ms = 0.0
    env_stage = [0.0, 0.0, 0.0]      # step / finishing kernel (caller's stream), event kernels, pre-solve (side stream)
    lib.cn_env_profile(env._h, 1)
    reps = 5
    for _ in range(reps):
        s = rollouts.step
        o = {k: rollouts.obs[k][s] for k in rollouts.obs}
        value, action, logp, h_new = eng.act(o, rollouts.recurrent_hidden_states['human_node_rnn'][s], rollouts.masks[s])
        buf = (C.c_float * ns)()
        _capi.check(lib, lib.cn_policy_stage_ms(eng._h, buf, ns), "stage_ms")
        for i in range(ns):
            acc[i] += buf[i] / reps
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        nobs, rew, done, info = env.step_device(action)
        g1.record()
        torch.cuda.synchronize()
        env_ms += g0.elapsed_time(g1) / reps
        ebuf = (C.c_float * 3)()
        _capi.check(lib, lib.cn_env_stage_ms(env._h, ebuf), "cn_env_stage_ms")
        for i in range(3):
            env_stage[i] += ebuf[i] / reps
        rollouts.insert(nobs, {'human_node_rnn': h_new}, action, logp, value, rew, (1.0 - done.float()).unsqueeze(1))
    lib.cn_policy_profile(eng._h, 0)
    lib.cn_env_profile(env._h, 0)
    stages = dict(zip(names, acc))
    rows_valid = int(lib.cn_policy_last_rows(eng._h))          # compacted human rows of the last act

    # ---------------------------------------------------------------- PPO update of the headline config (all-reduce active)
    update_c2 = None
    if not a.no_update:
        while rollouts.step != 0:
            device_step()
        for _ in range(ROLLOUT_T):
            device_step()                          # a fresh 30-step rollout; after_update ran at the boundary
        update_c2 = _ppo_update_block(torch, policy, rollouts, world, N)

    # ---------------------------------------------------------------- the shipped checkpoint as the load (if it is on the box)
    shipped = None
    ck = os.path.join(REPO, "local_ckpt", "41665.pt")
    if os.path.exists(ck) and not a.no_update:
        policy.load_state_dict(torch.load(ck, map_location=dev, weights_only=True))
        for _ in range(200):
            device_step()
        barrier()
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0.record()
        for _ in range(a.steps):
            device_step()
        h1.record()
        barrier()
        shipped = {"ms_total": h0.elapsed_time(h1), "rows": int(lib.cn_policy_last_rows(eng._h))}

    # ---------------------------------------------------------------- the other BASELINE configs (c3, c4, c5)
    env.close()
    del eng, rollouts, env
    policy._cuda = None
    torch.cuda.empty_cache()
    extra = {}
    names_extra = [c for c in a.configs.split(",") if c in EXTRA_CONFIGS]
    for c in names_extra:
        extra[c] = _run_extra_config(torch, dist, c, EXTRA_CONFIGS[c], dev, rank, world, a.config_steps, 5, a.config_burn_in,
                                     with_update=not a.no_update)

    # max over ranks
    vec = [ms_value, ms_e2e, wall_e2e, update_c2["ms"] if update_c2 else 0.0, update_c2["allreduce_ms"] if update_c2 else 0.0,
           shipped["ms_total"] if shipped else 0.0]
    for c in names_extra:
        vec += [extra[c]["ms_total"], extra[c].get("update", {}).get("ms", 0.0), extra[c].get("update", {}).get("allreduce_ms", 0.0)]
    t = torch.tensor(vec, device=dev, dtype=torch.float64)
    cnt = torch.tensor([float(extra[c]["spawn_overflow_envs"]) for c in names_extra] + [0.0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    vec = [float(x) for x in t]
    ms_value, ms_e2e, wall_e2e = vec[0:3]
    if update_c2:
        update_c2["ms"], update_c2["allreduce_ms"] = vec[3], vec[4]
        update_c2["allreduce_share"] = vec[4] / vec[3] if vec[3] > 0 else None
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    total_envs = N * world
    value = total_envs * a.steps / (ms_value / 1000.0)
    e2e_ms = max(ms_e2e, wall_e2e)
    e2e = total_envs * a.steps / (e2e_ms / 1000.0)
    peaks = {}
    pk = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks = json.load(open(pk))
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)" if peaks else \
        "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"
    hbm = peaks.get("hbm_gbs", 6650.0)
    # QKV projection: algorithmic FLOPs of ONE launch = 2 * rows * 1536 * 512 over the rows actually
    # processed (padded humans are compacted out; the dense row count is reported next to it)
    qkv_flops = 2.0 * rows_valid * 1536 * 512
    qkv_ms = stages.get("qkv_gemm", 0.0)
    qkv_tf = qkv_flops / (qkv_ms / 1000.0) / 1e12 if qkv_ms > 0 else 0.0
    gemm_kernel = "cn_gemm_tc_kernel (tcgen05 3xFP16)" if a.gemm_mode == 1 else "cn_gemm_f32_kernel"
    roof_gemm = {"kernel": "%s QKV projection, rows=%d N=1536 K=512" % (gemm_kernel, rows_valid), "bound": "tensor",
                 "achieved": qkv_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": qkv_tf / peak_tf if peak_tf else None,
                 "traffic": None, "peak_source": peak_src, "launch_ms": qkv_ms, "algorithmic_flops_per_launch": qkv_flops,
                 "mma_flops_issued_per_launch": qkv_flops * (3 if a.gemm_mode == 1 else 1), "dense_rows": N * HUMANS}
    # environment step: algorithmic bytes per launch = B_env * N (SURVEY.md §8d) / CUDA-event time
    # The step is TWO launches of cn_env_step_kernel since round 2: the ORCA solve of all humans runs ahead on the side
    # stream (pre-solve, timed alone here: nothing else is enqueued while the profiling loop waits), the launch on the
    # caller's stream only finishes the step.  Their CUDA-event durations are added.
    env_ms = env_stage[0] + env_stage[2]
    env_gbs = B_ENV * N / (env_ms / 1000.0) / 1e9 if env_ms > 0 else 0.0
    # dram__bytes_read.sum + dram__bytes_write.sum of the two launches at N=4096, H=20 (ncu --set full of the final code,
    # profiles/r2_env_step_presolve_ncu_raw.csv): pre-solve 8.26 MB + 0.33 MB, finishing pass 8.30 MB + 0.01 MB -- the
    # state is read twice since the solve runs ahead, 1.4x the algorithmic bytes
    env_traffic = 16.90e6 * N / 4096.0 if HUMANS == 20 else None
    roof_env = {"kernel": "cn_env_step_kernel, pre-solve launch (side stream, %.4f ms) + finishing launch (%.4f ms): one rollout "
                          "step of %d envs; cn_env_event_kernel runs on the side stream" % (env_stage[2], env_stage[0], N),
                "bound": "hbm",
                "achieved": env_gbs, "peak": hbm, "unit": "GB/s", "frac": env_gbs / hbm, "traffic": env_traffic,
                "traffic_source": "ncu --set full capture profiles/r2_env_step_presolve_ncu_raw.csv (both launches), scaled by N/4096",
                "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6.65 TB/s", "launch_ms": env_ms,
                "algorithmic_bytes_per_launch": B_ENV * N,
                "note": "latency/divergence bound by construction (per-human ORCA LP), see DESIGN.md"}
    dominant_is_env = env_ms >= max(stages.values())
    per_gpu_gbs = value / world * (B_ENV + B_POL) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms_value / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "CrowdSimPred-v0 const_vel, 20 humans, HH+HR attention, %d envs per GPU (BASELINE configs[1])" % N,
                   "global_envs": total_envs, "rollout_T": ROLLOUT_T, "parallelism": "env-sharded dp%d" % world,
                   "weights": "random init (orthogonal), seed 425", "gemm_mode": a.gemm_mode,
                   "burn_in_steps": a.burn_in, "host_affinity": affinity,
                   "state": "desynchronised steady state (episodes at mixed phases, auto-resets every step); the "
                            "lock-step first episodes right after reset() cost up to 0.69 ms/step (profiles/r1_step_series.json)",
                   "l2": "no flush: every step touches a different rollout-storage slot (30 slots x 4.3 MB of observations) plus ~170 MB of policy activations and 19 MB of env state, > the 126 MB L2"},
        "e2e": {"value": e2e, "unit": UNIT,
                "h2d_bytes_per_step": N * 4 * 3,                 # masks + bad_masks + reward into the storage
                "d2h_bytes_per_step": N * (4 + 1 + 4 + 4 + 8 + 4),   # reward, done, info, aux, ep_ret, ep_len
                "ms_per_step": e2e_ms / a.steps, "ms_per_step_cuda_events": ms_e2e / a.steps},
        "gpu_launches": int(launches), "cpu_enqueue_ms_per_step": cpu_enqueue_ms,
        "roofline": roof_env if dominant_is_env else roof_gemm,
        "roofline_other": roof_gemm if dominant_is_env else roof_env,
        "valid_human_rows": rows_valid, "mean_detected_humans": rows_valid / float(N),
        "breakdown_ms": {"env_step_kernel": env_stage[0], "env_presolve_kernel_side_stream": env_stage[2],
                         "env_event_kernels_side_stream": env_stage[1], **stages},
        "hbm_roofline": {"bytes_per_env_step": B_ENV + B_POL, "achieved_gbs_per_gpu": per_gpu_gbs,
                         "peak_gbs_per_gpu": hbm, "frac": per_gpu_gbs / hbm,
                         "note": "per GPU: whole-job env-steps/s / n_gpus x algorithmic bytes per env-step (SURVEY.md 8d) "
                                 "against ONE GPU's measured copy bandwidth"},
        "clocks": clocks,
    }
    if update_c2:
        it_ms = ROLLOUT_T * ms_value / a.steps + update_c2["ms"]
        line["update"] = dict(update_c2, whole_loop_env_steps_per_s=total_envs * ROLLOUT_T / (it_ms / 1000.0),
                              note="one training iteration = 30 rollout steps + GAE + this update; the metric `value` is the "
                                   "rollout phase alone (SURVEY.md 8d)")
    if shipped:
        line["shipped_checkpoint"] = {"weights": "trained_models/GST_predictor_rand/checkpoints/41665.pt (local_ckpt/)",
                                      "value": total_envs * a.steps / (vec[5] / 1000.0), "ms_per_step": vec[5] / a.steps,
                                      "mean_detected_humans": shipped["rows"] / float(N)}
    cfgs = {}
    off = 6
    for i, c in enumerate(names_extra):
        spec, ex = EXTRA_CONFIGS[c], extra[c]
        ms_c, up_ms, ar_ms = vec[off + 3 * i], vec[off + 3 * i + 1], vec[off + 3 * i + 2]
        envs_total = spec["envs"] * world
        d = {"workload": spec["workload"], "humans": spec["H"], "envs_per_gpu": spec["envs"], "global_envs": envs_total,
             "steps": a.config_steps, "burn_in_steps": a.config_burn_in, "ms_per_step": ms_c / a.config_steps,
             "env_steps_per_s": envs_total * a.config_steps / (ms_c / 1000.0), "gpu_launches": ex["launches"],
             "mean_detected_humans": ex["valid_human_rows"] / float(spec["envs"]),
             "spawn_overflow_envs": int(cnt[i]), "deferred_events_rank0": ex["deferred_events"]}
        if "update" in ex:
            d["update"] = dict(ex["update"], ms=up_ms, allreduce_ms=ar_ms, allreduce_share=ar_ms / up_ms if up_ms > 0 else None)
        cfgs[c] = d
    if cfgs:
        line["configs"] = cfgs
    if world == 1 and not a.no_cpu_baseline:
        # bounded sample (~a.cpu_seconds of wall time) in a CHILD process: the reference's modules (rl, crowd_sim) and
        # its fork workers stay out of this process
        try:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps",
                                  str(max(4, int(a.cpu_seconds / 0.06))), "--warmup", "2"], capture_output=True, text=True,
                                 timeout=600, cwd=REPO)
            ref_line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
            line["cpu_baseline"] = ref_line["cpu_baseline"]
        except Exception as e:      # the baseline is a reported number, never a reason to lose the bench line
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": repr(e)[:300]}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
