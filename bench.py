#!/usr/bin/env python
"""bench.py -- headline benchmark of the rollout hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's algorithm on host cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as .npy

Workload (BASELINE.json configs[1], SURVEY.md section 8d "cfg 2"): random-action step throughput,
vs_dummy / hard difficulty, max_episode_steps=500, `--envs-per-gpu` envs per GPU (default
1 048 576), fp32 observations as the reference API specifies, auto-reset on done. A "step" is one
fused step+obs kernel launch over the whole batch. P1 action ids are pre-generated uniformly on
0..12 (16 int8 arrays resident in HBM, cycled); synthetic data, no dataset involved.

Prints ONE JSON line (rank 0). Keys: see the task contract; `roofline` = fused step kernel vs the
measured HBM copy peak; `cpu_baseline` = the oracle port timed on this box's host cores;
`e2e` = the same metric through the host-buffer C-ABI call (inv_step_host) with the action upload
and the full observation/reward/done download inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
N_ACTION_SETS = 16


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)   # SURVEY.md section 8d: 1000 timed steps ...
    ap.add_argument("--warmup", type=int, default=600)   # ... after 600 warm-up steps (past the first timeout)
    ap.add_argument("--preroll", type=int, default=-1,
                    help="untimed steps BEFORE the warm-up, so that the timed steps lie past the first episode timeout "
                         "(SURVEY 8(d)) whatever --warmup says; -1 = max(0, max_episode_steps + 100 - warmup)")
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--envs-per-gpu", type=int, default=1 << 20)
    ap.add_argument("--obs-dtype", choices=["f32", "bf16", "u8"], default="f32")
    ap.add_argument("--mode", choices=["dummy", "selfplay"], default="dummy")
    ap.add_argument("--difficulty", choices=["easy", "hard"], default="hard")
    ap.add_argument("--max-episode-steps", type=int, default=500)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=8, help="timed host-buffer steps (0 = skip e2e)")
    ap.add_argument("--e2e-envs", type=int, default=0, help="envs per GPU for the e2e leg (0 = same as --envs-per-gpu)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg (0 = skip)")
    ap.add_argument("--cpu-sample-envs", type=int, default=65536)
    ap.add_argument("--sweep", action="store_true", help="also time 4K..4M envs (written to stderr)")
    ap.add_argument("--ppo", type=int, default=1, help="1 = also run the PPO block (BASELINE.json configs[3]/[4]), 0 = skip")
    ap.add_argument("--ppo-envs3", type=int, default=65536, help="envs per GPU of the selfplay PPO run (configs[3])")
    ap.add_argument("--ppo-envs4", type=int, default=1 << 20, help="envs per GPU of the sharded vs_dummy PPO run (configs[4])")
    ap.add_argument("--ppo-samples", type=int, default=1 << 21, help="samples per GPU per PPO iteration (rollout_steps = this / envs)")
    ap.add_argument("--ppo-iters", type=int, default=3, help="PPO iterations per run (the first one is warm-up)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (a fixed sample of "
                         "the envs), so that two builds can be compared output for output; bench_outputs/ is git-ignored")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 arm; it does not apply to --impl reference")
    return args


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_tflops():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    except Exception:
        return 1400.0, "fallback (B200_PROFILING.md: ~1.4 PFLOP/s sustained)"


POLICY_FWD_FLOP = 92.6e6  # conv1..4 (3x3, 12-32-64-128-128 on 15x10) + the two 19204x256 heads, multiply-add = 2


def ppo_block(args, rank, world, dev):
    """PPO samples/s, the second half of BASELINE.json's metric, on its two policy-driven configs:
    configs[3] selfplay (both players policy-driven, batched bf16 inference + fused step) and
    configs[4] env-sharded vs_dummy/hard PPO with the NCCL gradient all-reduce. Both run the
    reference's update schedule (4 epochs over every sample, ppo_agent.py:19-27 / :190-231) through
    the repo's own trainer (inversus_b200.training.train). The rollout is cut to `--ppo-samples`
    samples per GPU per iteration so the block fits the bench budget (the reference collects 128
    steps per env, training.py:105-107; per-sample cost does not depend on that length) -- the
    line states the rollout length used. One extra run with epochs=1 is labelled as such."""
    import tempfile
    import torch
    import torch.distributed as dist
    from inversus_b200.training import train

    peak_tf, peak_src = measured_tflops()

    def run(name, mode, envs_per_gpu, epochs, iters):
        n_total = envs_per_gpu * world
        T = max(2, args.ppo_samples // envs_per_gpu)
        batch = 32768 if envs_per_gpu * T >= (1 << 19) else 16384
        torch.manual_seed(args.seed)
        with tempfile.TemporaryDirectory() as tmp:
            out = train(mode, n_total, total_steps=n_total * T * iters, log_dir=tmp,
                        opponent_difficulty="hard", precision="bf16", rollout_steps=T, batch_size=batch, epochs=epochs,
                        seed=args.seed, quiet=True, save=False, time_allreduce=True)
        st = out["steady_state"]
        # every rank times its own iterations; collectives keep them in step, report the slowest
        t = torch.tensor([st["rollout_s"], st["update_s"]], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        roll_s, upd_s = t.tolist()
        n = st["samples"]  # whole-job samples in the timed iterations
        infer_flop = POLICY_FWD_FLOP * n * (2 if mode == "selfplay" else 1)
        infer_flop += POLICY_FWD_FLOP * n_total * st["iterations"]  # the bootstrap value pass after each rollout
        upd_flop = 3 * POLICY_FWD_FLOP * n * epochs
        r = {"run": name, "mode": mode, "envs_per_gpu": envs_per_gpu, "total_envs": n_total, "rollout_steps": T,
             "epochs": epochs, "batch_size_per_gpu": batch, "iterations_timed": st["iterations"],
             "samples_per_s": n / (roll_s + upd_s),
             "rollout_env_steps_per_s": n / roll_s,
             "update_samples_per_s": n * epochs / upd_s,
             "rollout_s": roll_s, "update_s": upd_s,
             "inference_tflops_per_gpu": infer_flop / roll_s / 1e12 / world,
             "update_tflops_per_gpu": upd_flop / upd_s / 1e12 / world,
             "inference_frac_of_bf16_sustained": infer_flop / roll_s / 1e12 / world / peak_tf,
             "update_frac_of_bf16_sustained": upd_flop / upd_s / 1e12 / world / peak_tf,
             "precision": "bf16", "packed_encoder": out.get("packed_encoder"), "cuda_graph_rollout": out.get("cuda_graph"),
             "allreduce": out.get("allreduce"),
             "policy_loss": out.get("policy_loss"), "value_loss": out.get("value_loss"), "entropy": out.get("entropy")}
        return r

    runs = [
        run("configs[3] selfplay, reference schedule (4 epochs)", "selfplay", args.ppo_envs3, 4, args.ppo_iters),
        run("configs[4] vs_dummy hard sharded, reference schedule (4 epochs)", "vs_dummy", args.ppo_envs4, 4, args.ppo_iters),
        run("configs[4] vs_dummy hard sharded, epochs=1 (NOT the reference schedule)", "vs_dummy", args.ppo_envs4, 1,
            args.ppo_iters),
    ]
    return {"metric": "ppo_samples_per_sec", "unit": "samples/s (whole job; rollout + update wall clock, max over ranks)",
            "bf16_peak_tflops": peak_tf, "peak_source": peak_src, "policy_fwd_flop_per_sample": POLICY_FWD_FLOP,
            "note": "update_samples_per_s counts every epoch's pass over a sample; TFLOP/s = 3 x fwd FLOPs per "
                    "sample-pass for the update, fwd FLOPs per policy evaluation for the rollout (env step, sampling "
                    "and rollout stores are inside rollout_s)",
            "runs": runs}


def recorded_traffic(obs_dtype, mode, n_envs):
    """dram bytes per launch from the committed ncu capture of this kernel (profiles/traffic.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        return t.get(f"{mode}_{obs_dtype}") if t.get("envs") == n_envs else None
    except Exception:
        return None


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, v in names.items():
                    if bits & v:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.005)

    def __enter__(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._t:
            self._t.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------
# CPU leg: the oracle port (oracle/inversus_oracle.c) on the host cores. Used as `cpu_baseline` of
# our own line and as the whole measurement of `--impl reference`. The reference itself is pure
# Python and cannot travel to the GPU box; SURVEY.md section 6 gives its own speed measured in the
# builder container (about 5e3 env-steps/s per core through MultiEnvRunner.step).
def run_oracle(args, n_envs, steps, warmup, budget_s=None):
    import numpy as np
    from oracle import oracle as orc
    cores = orc.lib().orc_max_threads()
    b = orc.OracleBatch(n_envs, args.mode, args.difficulty, args.max_episode_steps, seed=args.seed, nthreads=cores)
    rs = np.random.RandomState(args.seed)
    acts = rs.randint(0, 13, size=(N_ACTION_SETS, n_envs)).astype(np.int8)
    acts2 = rs.randint(0, 13, size=(N_ACTION_SETS, n_envs)).astype(np.int8) if args.mode == "selfplay" else None
    b.reset()

    def one(t):
        b.step(acts[t % N_ACTION_SETS], None if acts2 is None else acts2[t % N_ACTION_SETS], auto_reset=True)
    for t in range(warmup):
        one(t)
    done_steps = 0
    t0 = time.perf_counter()
    for t in range(steps):
        one(warmup + t)
        done_steps += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return {"value": n_envs * done_steps / dt, "seconds": dt, "steps": done_steps, "cores": cores}


def run_reference_loop(args, seconds=4.0, n_envs=64):
    """The reference's OWN Python step loop -- MultiEnvRunner.step (inversus_rl/env_wrappers.py:485-528)
    plus the trainer's reset-on-done (inversus_rl/training.py:140-151) -- from the unmodified files
    staged under oracle/_ref by oracle/make_ref.sh, timed on ONE host core. Returns None when the
    staged copy is absent or the mode needs a policy callback (selfplay)."""
    ref = os.path.join(ROOT, "oracle", "_ref")
    if args.mode != "dummy" or not os.path.exists(os.path.join(ref, "inversus_rl", "env_wrappers.py")):
        return None
    import numpy as np
    sys.path.insert(0, ref)
    try:
        from inversus_rl.env_wrappers import MultiEnvRunner  # the reference's module, not this repo's
    finally:
        sys.path.remove(ref)
    runner = MultiEnvRunner(n_envs, "dummy", args.difficulty, args.max_episode_steps, seed=args.seed)
    rs = np.random.RandomState(args.seed)
    acts = rs.randint(0, 13, size=(64, n_envs))
    runner.reset()

    def one(k):
        (grid, extra), _, dones, _ = runner.step(acts[k % 64])
        for i in np.nonzero(dones)[0]:
            g, e = runner.envs[i].reset()
            grid[i], extra[i] = g, e
    for k in range(3):
        one(k)
    t0 = time.perf_counter()
    k = 0
    while time.perf_counter() - t0 < seconds:
        one(k)
        k += 1
    dt = time.perf_counter() - t0
    try:
        commit = open(os.path.join(ref, "SOURCE_COMMIT")).read().strip()
    except OSError:
        commit = "unknown"
    return {"value": n_envs * k / dt, "unit": UNIT, "cores": 1, "kind": "reference",
            "sample": f"{n_envs} envs x {k} steps ({dt:.1f} s), the reference's MultiEnvRunner.step + trainer-style "
                      f"reset-on-done, unmodified files staged by oracle/make_ref.sh (commit {commit[:12]}), "
                      f"stdlib Mersenne Twister draws, fp32 obs built every step"}


def run_python_loop(args, seconds=4.0, n_envs=64):
    """The reference's PYTHON step loop, restated in oracle/py_loop.py with the reference's own data
    structures (pinned to the golden fixtures), timed on ONE host core: the number the north star
    asks to see beside the GPU result. The live reference measured 6.0e3 env-steps/s on one core of
    the builder container where this restatement measured 7.7e3."""
    got = run_reference_loop(args, seconds, n_envs)
    if got is not None:
        return got
    import numpy as np
    from oracle.py_loop import PyRunner
    r = PyRunner(n_envs, args.mode, args.difficulty, args.max_episode_steps, seed=args.seed)
    rs = np.random.RandomState(args.seed)
    acts = rs.randint(0, 13, size=(64, n_envs))
    acts2 = rs.randint(0, 13, size=(64, n_envs)) if args.mode == "selfplay" else None
    r.reset()
    for t in range(3):
        r.step(acts[t], None if acts2 is None else acts2[t], None, auto_reset=True)
    t0 = time.perf_counter()
    k = 0
    while time.perf_counter() - t0 < seconds:
        r.step(acts[k % 64], None if acts2 is None else acts2[k % 64], None, auto_reset=True)
        k += 1
    dt = time.perf_counter() - t0
    return {"value": n_envs * k / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"{n_envs} envs x {k} steps ({dt:.1f} s), MultiEnvRunner-style sequential Python loop "
                      f"(oracle/py_loop.py), fp32 obs built every step, auto-reset"}


def _ref_worker(ref_dir, n_envs, mode, difficulty, max_steps, seed, warmup, steps, barrier, out_q):
    """One process of the reference arm: the staged reference's MultiEnvRunner, stepped like its trainer does."""
    import numpy as np
    sys.path.insert(0, ref_dir)
    from inversus_rl.env_wrappers import MultiEnvRunner
    runner = MultiEnvRunner(n_envs, mode, difficulty, max_steps, seed=seed)
    rs = np.random.RandomState(seed)
    acts = rs.randint(0, 13, size=(64, n_envs))
    runner.reset()

    def one(k):
        (grid, extra), _, dones, _ = runner.step(acts[k % 64])
        for i in np.nonzero(dones)[0]:  # inversus_rl/training.py:140-151
            g, e = runner.envs[i].reset()
            grid[i], extra[i] = g, e
    for k in range(warmup):
        one(k)
    barrier.wait()
    t0 = time.perf_counter()
    for k in range(steps):
        one(warmup + k)
    out_q.put(time.perf_counter() - t0)


def run_reference_processes(args, warmup, steps, envs_per_proc=64):
    """The unmodified reference (oracle/_ref) on ALL host cores: one process per core, each with its own
    MultiEnvRunner over `envs_per_proc` envs. Returns None if the staged copy is missing."""
    ref = os.path.join(ROOT, "oracle", "_ref")
    if args.mode != "dummy" or not os.path.exists(os.path.join(ref, "inversus_rl", "env_wrappers.py")):
        return None
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    cores = max(1, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    barrier, q = ctx.Barrier(cores + 1), ctx.Queue()
    procs = [ctx.Process(target=_ref_worker, args=(ref, envs_per_proc, "dummy", args.difficulty, args.max_episode_steps,
                                                   args.seed + 1000 * i, warmup, steps, barrier, q)) for i in range(cores)]
    for p in procs:
        p.start()
    barrier.wait()
    t0 = time.perf_counter()
    times = [q.get() for _ in procs]
    dt = time.perf_counter() - t0
    for p in procs:
        p.join()
    return {"value": cores * envs_per_proc * steps / dt, "seconds": dt, "steps": steps, "cores": cores,
            "envs": cores * envs_per_proc, "slowest_worker_s": max(times)}


def reference_arm(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return 0
    W = min(max(args.warmup, 3), 50)
    # the CPU arm has no caches or clocks to settle: its warm-up is capped, and each "step" is one
    # MultiEnvRunner.step over a bounded sample of the workload's envs (64 per host core). Both legs
    # time exactly --steps steps.
    ref = run_reference_processes(args, W, args.steps)
    n = args.cpu_sample_envs
    port = run_oracle(args, n, args.steps, W)
    port_line = {"value": port["value"], "unit": UNIT, "cores": port["cores"], "kind": "port",
                 "sample": f"{n} envs x {port['steps']} steps through oracle/inversus_oracle.c (the C restatement), "
                           f"fp32 obs written every step, auto-reset, {port['cores']} pthreads"}
    if ref:
        r, kind = ref, "reference"
        sample = (f"{ref['envs']} envs ({ref['cores']} processes x 64) x {ref['steps']} steps of the same workload through the "
                  f"reference's own MultiEnvRunner.step + reset-on-done (unmodified files staged by oracle/make_ref.sh), "
                  f"fp32 obs built every step, one process per host core")
    else:
        r, kind, sample = port, "port", port_line["sample"]
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": W, "ms_per_step": 1e3 * r["seconds"] / max(r["steps"], 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": workload_config(args, max(args.gpus, 1)),   # the B200 arm's config at this N, key for key
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": kind, "sample": sample},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "c_port": port_line,
        "gpu_launches": 0,
        "note": "kind=reference: the reference's pure-Python step loop itself, on every host core of this box. "
                "c_port: the same algorithm restated in C (oracle/inversus_oracle.c), for scale.",
    }
    emit(line)
    return 0


def resolved_preroll(args):
    """Untimed steps before the warm-up (a function of the flags only, so both arms print the same config)."""
    return args.preroll if args.preroll >= 0 else max(0, args.max_episode_steps + 100 - max(args.warmup, 3))


def workload_config(args, world):
    return {
        "workload": f"random-action fused step+obs, vs_{args.mode} {args.difficulty}, "
                    f"{args.envs_per_gpu} envs/GPU, max_episode_steps={args.max_episode_steps} "
                    f"(BASELINE.json configs[1])",
        "envs_per_gpu": args.envs_per_gpu, "total_envs": args.envs_per_gpu * world,
        "mode": args.mode, "difficulty": args.difficulty, "max_episode_steps": args.max_episode_steps,
        "obs_dtype": args.obs_dtype, "auto_reset": True,
        "preroll_steps": resolved_preroll(args),
        "regime": "timed steps start after preroll + warmup steps, past the first episode timeout (desynchronised episodes)",
        "actions": f"pre-generated uniform int8 ids, {N_ACTION_SETS} arrays in HBM cycled",
        "parallelism": f"env-sharded x{world}, no collective in the step path",
        "l2": "per-step working set (obs write stream, 7.2 KB/env) far exceeds the 126 MB L2; no explicit flush",
    }


def time_steps(sim, torch, acts, acts2, steps, first_t=0):
    """K back-to-back launches; returns per-launch ms measured with CUDA events on the launch stream."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for t in range(steps):
        k = (first_t + t) % N_ACTION_SETS
        sim.step(acts[k], None if acts2 is None else acts2[k])
        ev[t + 1].record()
    torch.cuda.synchronize()
    return [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)], ev[0].elapsed_time(ev[steps])


DUMP_ENVS = 1 << 18      # envs whose per-env outputs are written (all of them up to this many)
DUMP_OBS_ENVS = 2048     # of those, envs whose observations are written (7.2 KB per view in fp32)
DUMP_SAMPLE_SEED = 12345


def dump_outputs(path, sim):
    """Writes what the last `sim.step` returned -- (obs, extra), reward, done, info, plus the episode
    statistics it leaves as attributes and, in selfplay, P2's view (obs_p2, extra_p2) -- as
    float32/float64 .npy files, for a fixed, seeded sample of the envs: at most about 47 MB whatever
    the env count and mode. env_index / obs_env_index name the sampled envs."""
    import numpy as np
    import torch
    pick = np.random.RandomState(DUMP_SAMPLE_SEED).permutation(sim.num_envs)[:DUMP_ENVS]
    rows, obs_rows = np.sort(pick), np.sort(pick[:DUMP_OBS_ENVS])
    idx = torch.from_numpy(rows).to(sim.device)
    obs_idx = torch.from_numpy(obs_rows).to(sim.device)
    arrays = {"env_index": rows.astype(np.float64), "obs_env_index": obs_rows.astype(np.float64)}
    outputs = [("obs", sim.obs, obs_idx, torch.float32), ("extra", sim.extra, idx, torch.float32),
               ("reward", sim.reward, idx, torch.float32), ("done", sim.done, idx, torch.float32),
               ("info", sim.info, idx, torch.float32), ("episode_steps", sim.episode_steps, idx, torch.float64),
               ("episode_return", sim.episode_return, idx, torch.float64)]
    if sim.obs_p2 is not None:
        outputs += [("obs_p2", sim.obs_p2, obs_idx, torch.float32), ("extra_p2", sim.extra_p2, idx, torch.float32)]
    for name, t, ix, dt in outputs:
        arrays[name] = t.index_select(0, ix).to(dt).cpu().numpy()
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


_REAL_STDOUT = None


def claim_stdout():
    """Keep stdout clean for the ONE JSON line: libraries (NCCL prints its version banner to fd 1)
    are redirected to stderr for the duration of the run."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


def main():
    args = parse_args()
    if args.impl == "reference":
        return reference_arm(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from inversus_b200 import BatchedInversus, constants
    from inversus_b200.sharding import dist_env

    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:  # convenience: relaunch under torchrun
        import subprocess
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29511", os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    claim_stdout()
    rank, local_rank, world = dist_env()
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(0)
    dev = torch.device("cuda", local_rank if world > 1 else 0)
    n = args.envs_per_gpu
    selfplay = args.mode == "selfplay"

    sim = BatchedInversus(n, args.mode, args.difficulty, args.max_episode_steps, seed=args.seed,
                          device=dev.index, obs_dtype=args.obs_dtype, auto_reset=True, env_id_base=rank * n)
    g = torch.Generator(device=dev)
    g.manual_seed(args.seed * 1000 + rank)
    acts = [torch.randint(0, 13, (n,), device=dev, dtype=torch.int8, generator=g) for _ in range(N_ACTION_SETS)]
    acts2 = [torch.randint(0, 13, (n,), device=dev, dtype=torch.int8, generator=g) for _ in range(N_ACTION_SETS)] if selfplay else None
    sim.reset()
    W = max(args.warmup, 3)
    # pre-roll: with a short --warmup every timed step would lie inside the synchronised first episodes
    # (all envs time out together at step 500); these untimed steps put the timed region in the steady,
    # desynchronised regime the metric is defined on. ~0.7 s at 1 M envs.
    preroll = resolved_preroll(args)
    for t in range(preroll + W):
        sim.step(acts[t % N_ACTION_SETS], None if acts2 is None else acts2[t % N_ACTION_SETS])
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ------------------------------------------------------------------ timed region (device)
    launches0 = sim.launch_count
    barrier()
    with ClockSampler(dev.index) as clk:
        per_launch_ms, total_ms = time_steps(sim, torch, acts, acts2, args.steps, preroll + W)
        barrier()
    launches = sim.launch_count - launches0
    status = sim.poll_status()
    assert status == 0, f"device status bits {status}"
    if args.dump_outputs and rank == 0:  # before the e2e leg steps the same envs again
        dump_outputs(args.dump_outputs, sim)
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    value = n * world * args.steps / (total_ms_max * 1e-3)

    # write-only ceiling of this GPU, measured live: the step kernel is 99 % stores, and a pure store
    # stream runs above the copy figure that MEASURED_PEAKS.json holds (no read/write turnaround)
    fill = torch.empty(1 << 30, dtype=torch.float32, device=dev)  # 4 GiB
    for _ in range(2):
        fill.zero_()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(5):
        fill.zero_()
    f1.record()
    torch.cuda.synchronize()
    fill_gbs = 5 * fill.numel() * 4 / (f0.elapsed_time(f1) * 1e-3) / 1e9
    del fill
    torch.cuda.empty_cache()

    elem = {"f32": 4, "bf16": 2, "u8": 1}[args.obs_dtype]
    alg_bytes = constants.algorithmic_bytes_per_env_step(elem, selfplay) * n
    avg_launch_ms = sum(per_launch_ms) / len(per_launch_ms)
    peak, peak_src = measured_peaks()
    achieved = alg_bytes / (avg_launch_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": recorded_traffic(args.obs_dtype, args.mode, n),
                "kernel": "inv::inv_kernel<OP_STEP> (fused step+obs)", "peak_source": peak_src,
                "write_only_ceiling_gbs": fill_gbs, "frac_of_write_only_ceiling": achieved / fill_gbs,
                "write_only_ceiling_source": "cudaMemset of 4 GiB timed in this run (the kernel's traffic is 99 % stores)",
                "algorithmic_bytes_per_launch": alg_bytes,
                "algorithmic_bytes_per_env_step": alg_bytes // n,
                "avg_launch_ms": avg_launch_ms, "min_launch_ms": min(per_launch_ms),
                "median_launch_ms": statistics.median(per_launch_ms)}

    # ------------------------------------------------------------------ e2e: host buffers through inv_step_host
    e2e = None
    e2e_variants = None
    esim = out = None
    if args.e2e_steps > 0:
        ne = args.e2e_envs or n
        esim = sim if ne == n else BatchedInversus(ne, args.mode, args.difficulty, args.max_episode_steps,
                                                   seed=args.seed, device=dev.index, obs_dtype=args.obs_dtype,
                                                   auto_reset=True, env_id_base=rank * ne)
        if esim is not sim:
            esim.reset()
        out = esim.host_buffers(pinned=True)
        rs = np.random.RandomState(args.seed + rank)
        pins = []

        def host_ids():  # action ids in page-locked host memory (they go to the device from there)
            t = torch.empty(ne, dtype=torch.int8, pin_memory=True)
            pins.append(t)
            a = t.numpy()
            a[:] = rs.randint(0, 13, size=ne)
            return a
        h_acts = [host_ids() for _ in range(4)]
        h_acts2 = [host_ids() for _ in range(4)] if selfplay else None
        views = 2 if selfplay else 1
        small = 4 + 1 + 1 + 4 + 8 + views * 16

        def run_e2e(nthreads, frac, with_obs, warm):
            esim.set_host_path(nthreads, frac)
            o = out if with_obs else {k: v for k, v in out.items() if not k.startswith("obs")}
            # a step without observations takes ~1.6 ms: time enough of them that one scheduling
            # hiccup on one of the ranks does not decide the max-over-ranks figure
            steps = args.e2e_steps if with_obs else max(50, 10 * args.e2e_steps)
            for k in range(warm if with_obs else max(warm, 10)):
                esim.step_host(h_acts[k % 4], None if h_acts2 is None else h_acts2[k % 4], o)
            barrier()
            t0 = time.perf_counter()
            for k in range(steps):
                esim.step_host(h_acts[k % 4], None if h_acts2 is None else h_acts2[k % 4], o)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
            hp = esim.host_path()
            if not with_obs:
                d2h = ne * small
            elif nthreads == 0 or args.obs_dtype != "f32" or ne < 4096:
                d2h = ne * (views * 1800 * elem + small)
            else:
                n_dma = int(hp["dma_fraction"] * ne)  # envs whose fp32 observation crosses PCIe as is
                d2h = ne * small + views * ((ne - n_dma) * 256 + n_dma * 7200)
            return {"value": ne * world * steps / dt, "unit": UNIT, "h2d_bytes_per_step": ne * views,
                    "d2h_bytes_per_step": d2h, "steps": steps, "envs_per_gpu": ne,
                    "ms_per_step": 1e3 * dt / steps, "host_threads": hp["threads"],
                    "dma_fraction": round(hp["dma_fraction"], 4)}

        # headline: every output of MultiEnvRunner.step, fp32 observations included, lands in host
        # buffers. Packed rows cross PCIe and are expanded on the host threads while the copy engine
        # moves the rest directly (inv_set_host_path, auto-balanced).
        local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))
        host_threads = max(1, min(32, (os.cpu_count() or 1) // max(local_world, 1)))  # ranks share the host cores
        e2e = run_e2e(host_threads, -1.0, True, warm=6)
        e2e["api"] = ("inv_step_host (C ABI), pinned host buffers: int8 action ids up; fp32 obs + extra + reward + done + "
                      "info + episode stats down (packed rows over PCIe + host-side expansion, balanced with direct DMA)")
        e2e_variants = {
            "plain_pcie_copy": run_e2e(0, 0.0, True, warm=1),
            "obs_stay_on_device": run_e2e(0, 0.0, False, warm=1),
        }
        e2e_variants["obs_stay_on_device"]["note"] = "actions up; reward/done/info/extra/episode stats down; observations consumed on the GPU"

        # the trainer's loop (training.py:140-151) with a GPU-resident policy: grid AND extra stay on the
        # device, reward/done/info arrive dense, episode statistics only for the episodes that ended
        def run_events():
            eo = esim.host_event_buffers(pinned=True)
            steps = max(50, 10 * args.e2e_steps)
            for k in range(10):
                esim.step_host_events(h_acts[k % 4], None if h_acts2 is None else h_acts2[k % 4], eo)
            barrier()
            finished = 0
            t0 = time.perf_counter()
            for k in range(steps):
                finished += len(esim.step_host_events(h_acts[k % 4], None if h_acts2 is None else h_acts2[k % 4], eo))
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
            per_step = finished / steps
            return {"value": ne * world * steps / dt, "unit": UNIT, "h2d_bytes_per_step": ne * views,
                    "d2h_bytes_per_step": int(ne * 6 + 8 + 24 * per_step), "steps": steps, "envs_per_gpu": ne,
                    "ms_per_step": 1e3 * dt / steps, "finished_episodes_per_step": per_step,
                    "api": "inv_step_host_events (C ABI)",
                    "note": "actions up; reward/done/info dense + one 24-byte record per finished episode down; "
                            "observations (grid and extra) consumed on the GPU"}
        e2e_variants["obs_stay_on_device_episode_events"] = run_events()
        esim.set_host_path(host_threads, -1.0)

    # ------------------------------------------------------------------ optional sweep (stderr)
    if args.sweep and rank == 0:
        for ns in (4096, 16384, 65536, 262144, 1048576, 4194304):
            s2 = BatchedInversus(ns, args.mode, args.difficulty, args.max_episode_steps, seed=args.seed,
                                 device=dev.index, obs_dtype=args.obs_dtype, auto_reset=True)
            a = [torch.randint(0, 13, (ns,), device=dev, dtype=torch.int8, generator=g) for _ in range(N_ACTION_SETS)]
            a2 = [torch.randint(0, 13, (ns,), device=dev, dtype=torch.int8, generator=g) for _ in range(N_ACTION_SETS)] if selfplay else None
            s2.reset()
            for t2 in range(50):
                s2.step(a[t2 % N_ACTION_SETS], None if a2 is None else a2[t2 % N_ACTION_SETS])
            torch.cuda.synchronize()
            pl, tot = time_steps(s2, torch, a, a2, 200)
            bts = constants.algorithmic_bytes_per_env_step(elem, selfplay) * ns
            # the same 16 steps captured once in a CUDA graph and replayed: launch overhead of the
            # Python/ctypes call path removed (what a graph-captured rollout loop would see)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for k in range(N_ACTION_SETS):
                    s2.step(a[k], None if a2 is None else a2[k])
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                for k in range(N_ACTION_SETS):
                    s2.step(a[k], None if a2 is None else a2[k])
            for _ in range(3):
                graph.replay()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = max(1, 400 // N_ACTION_SETS)
            e0.record()
            for _ in range(reps):
                graph.replay()
            e1.record()
            torch.cuda.synchronize()
            gms = e0.elapsed_time(e1) / (reps * N_ACTION_SETS)
            print(json.dumps({"sweep_envs": ns, "env_steps_per_sec": ns * 200 / (tot * 1e-3),
                              "ms_per_step": tot / 200, "hbm_gbs": bts / (tot / 200 * 1e-3) / 1e9,
                              "frac_of_peak": bts / (tot / 200 * 1e-3) / 1e9 / peak,
                              "cuda_graph": {"ms_per_step": gms, "env_steps_per_sec": ns / (gms * 1e-3),
                                             "frac_of_peak": bts / (gms * 1e-3) / 1e9 / peak}}),
                  file=sys.stderr, flush=True)
            del graph
            s2.close()
            del s2, a, a2

    # ------------------------------------------------------------------ cpu baseline (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and args.cpu_seconds > 0:
        nc = args.cpu_sample_envs
        r = run_oracle(args, nc, 10 ** 9, 3, budget_s=args.cpu_seconds)
        port = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                "sample": f"{nc} envs x {r['steps']} steps ({r['seconds']:.1f} s) of the same workload through "
                          f"oracle/inversus_oracle.c, fp32 obs written every step, {r['cores']} pthreads"}
        # the reference itself (unmodified Python, oracle/_ref) on every host core: ~15 ms per step of 64 envs per core
        ref = run_reference_processes(args, 5, max(20, int(args.cpu_seconds / 0.016)))
        if ref:
            cpu = {"value": ref["value"], "unit": UNIT, "cores": ref["cores"], "kind": "reference",
                   "sample": f"{ref['envs']} envs ({ref['cores']} processes x 64) x {ref['steps']} steps ({ref['seconds']:.1f} s) of "
                             f"the same workload through the reference's own MultiEnvRunner.step + reset-on-done "
                             f"(unmodified files staged by oracle/make_ref.sh), one process per host core",
                   "c_port": port}
        else:
            cpu = dict(port)
        cpu["python_loop"] = run_python_loop(args, seconds=min(4.0, args.cpu_seconds))

    # ------------------------------------------------------------------ PPO block (all ranks)
    ppo = None
    if args.ppo:
        sim.close()
        sim = esim = out = acts = acts2 = None  # device buffers and the pinned host buffers of the e2e leg
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        ppo = ppo_block(args, rank, world, dev)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W,
            "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32", "data": "synthetic", "config": workload_config(args, world),
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "e2e_variants": e2e_variants, "gpu_launches": launches,
            "clocks": clk.summary(), "ppo": ppo,
        }
        emit(line)
    if world > 1:
        shutdown_distributed(torch, dist, dev)
    return 0


def shutdown_distributed(torch, dist, dev):
    """Leave a torchrun job without hanging: the PPO block replays CUDA graphs that contain NCCL
    kernels, and tearing the communicator down while such graphs (or the watchdog's view of them)
    are alive has been seen to block forever. Drop the graphs, synchronise, give the orderly
    teardown 20 s on a side thread, then exit this worker with status 0."""
    import gc
    gc.collect()
    torch.cuda.synchronize(dev)
    dist.barrier()
    t = threading.Thread(target=dist.destroy_process_group, daemon=True)
    t.start()
    t.join(20.0)
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


if __name__ == "__main__":
    sys.exit(main())
