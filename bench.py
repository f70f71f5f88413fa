#!/usr/bin/env python
"""bench.py -- candidate action-sequences/sec of the PETS HalfCheetah CEM planning loop (BASELINE.json).

One "step" = one full CEM plan, i.e. one ``TrajectoryOptimizerAgent.act()`` worth of work: 5 iterations x
population 500 candidate sequences, each rolled out for H = 30 steps with 20 particles through the ensemble
(7 members, 5 elites, 4 x 200 SiLU).  ``value`` times it device-resident (inputs in HBM, CUDA events);
``e2e`` times the public API call ``agent.act(obs)`` with a host observation in and the host plan out.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

``--dump-outputs DIR``: after the timed steps, the plan the last timed step returned (``CEMOptimizer.optimize``'s
[H, A] solution, what ``agent.act`` hands back) is written to ``DIR/solution.npy`` (float32).  Every input is seeded
(model weights, observation, the optimiser's and the model's random streams), so two runs with the same arguments
plan from identical inputs and two builds can be compared output for output.

N > 1 (under torchrun): weak scaling -- every rank plans over its own 500-sequence shard of a 500 x N
population, ONE all-gather of local top-k records per CEM iteration (mbrl_lib_b200.dist); ``e2e`` is then
``ShardedCEMOptimizer.optimize`` per call with the host observation in and the host plan out, max over ranks.
The same run also reports BASELINE config 5 (fixed global populations 8 000 ... 64 000 sharded over the N GPUs,
strong scaling) with the collective's share of an iteration, in ``config5_population_scan_sharded``.

``--impl reference``: the UNMODIFIED reference (mbrl-lib from ``oracle/_ref``) timed on the host CPUs through
its own ``TrajectoryOptimizerAgent.act`` (rank 0 only); the oracle port is the fallback when it cannot be imported.
"""
import argparse
import csv
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from mbrl_lib_b200 import synthetic as syn  # noqa: E402

WORKLOAD = "halfcheetah"  # BASELINE.json configs[1]
CEM_ITERS, ELITE_RATIO, ALPHA = 5, 0.1, 0.1
FLOP_PER_SEQ = 157.68e6  # SURVEY.md section 8d: 2 * sum K*N (true dims) * P * H = 262 800 * 20 * 30
METRIC = "candidate action-sequences/sec, PETS HalfCheetah CEM"
# identical on both arms (ours and --impl reference): what is computed per step
CONFIG = {
    "workload": ("PETS gym___HalfCheetah-v4 dims (obs 17, act 6): ensemble 7 (5 elites) x 4x200 SiLU, CEM pop 500 x 5 iterations "
                 "per plan, horizon 30, 20 particles, TS1"),
    "step": "one 5-iteration CEM plan = one TrajectoryOptimizerAgent.act(): 2 500 candidate sequences per GPU",
}
NCU_SUMMARIES = ["profiles/r2_rollout_tc_ncu_full_summary.csv", "profiles/r1_rollout_tc_final_ncu_full_summary.csv"]


def measured_peak_tflops():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["bf16_tflops"]), "measured (MEASURED_PEAKS.json bf16_tflops, burst)"
    return 1590.0, "fallback (B200_PROFILING.md 1.59 PFLOP/s)"


def ncu_dram_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE rollout launch from the newest committed ncu --set full summary."""
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for rel in NCU_SUMMARIES:
        path = os.path.join(ROOT, rel)
        if not os.path.exists(path):
            continue
        tot, seen = 0.0, 0
        for row in csv.reader(open(path)):
            if len(row) >= 3 and row[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and row[1] in unit:
                tot += float(row[2]) * unit[row[1]]
                seen += 1
        if seen == 2:
            return int(tot), rel
    return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(len(r) > 2 + j and r[2 + j] == "Active" for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


class _Box:
    def __init__(self, lo, hi, n):
        self.low, self.high, self.shape = np.full(n, lo, np.float32), np.full(n, hi, np.float32), (n,)


def build_problem(device, workload=WORKLOAD, ts1="tile_shuffle"):
    import mbrl_lib_b200 as bp
    from mbrl_lib_b200 import functions

    spec = syn.CASES[workload]
    arrays = syn.make_model_arrays(spec)
    model = bp.model_from_arrays(spec, arrays, device)

    class _Env:
        observation_space = _Box(-np.inf, np.inf, spec.obs_dim)
        action_space = _Box(spec.action_lb, spec.action_ub, spec.act_dim)

    rew = functions.REWARD_FNS[spec.reward_fn] if spec.reward_fn else None
    env = bp.ModelEnv(_Env(), model, functions.TERM_FNS[spec.term_fn], rew,
                      generator=torch.Generator(device=device).manual_seed(0), precision="auto", ts1=ts1)
    return spec, arrays, env


def l2_flush_buffer(device):
    return torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=device)


def time_events(fn, reps, flush=None):
    """mean ms per call of fn() over `reps` calls, each bracketed by CUDA events (L2 flushed, untimed, before each)."""
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tot = 0.0
    for _ in range(reps):
        if flush is not None:
            flush.fill_(1)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        tot += s.elapsed_time(e)
    return tot / reps


def mbpo_step_extra(device, flush):
    """BASELINE config 4: ModelEnv.step over 100 000 start states x 1 step (MBPO rollouts), device-resident and
    through the reference-shaped numpy API (host arrays in, host arrays out)."""
    spec, _, env = build_problem(device, "mbpo_halfcheetah")
    B = 100000
    inp = syn.make_step_inputs(spec, B)
    state = env.reset(inp["obs"], return_as_np=False)
    act = torch.from_numpy(inp["act"]).to(device)
    for _ in range(3):
        env.step(act, state, sample=True)
    ms = time_events(lambda: env.step(act, state, sample=True), 10, flush)
    # numpy in / numpy out, as mbpo.py:31-63 calls it
    env.reset(inp["obs"], return_as_np=True)
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        st = env.reset(inp["obs"], return_as_np=True)
        env.step(inp["act"], st, sample=True)
    host_ms = (time.perf_counter() - t0) / reps * 1e3
    bytes_io = B * ((spec.obs_dim + spec.act_dim) * 4 + (spec.obs_dim + 1) * 4 + 1)
    return {"workload": "MBPO HalfCheetah: 100 000 start states x 1 model step (ModelEnv.step, ensemble 7, learned reward)",
            "device_resident_ms": ms, "device_resident_transitions_per_s": B / (ms * 1e-3),
            "numpy_api_ms": host_ms, "numpy_api_transitions_per_s": B / (host_ms * 1e-3),
            "numpy_api_bytes_over_pcie": bytes_io,
            "flop_per_transition": 263600}


def build_problem_variant(device, workload, **over):
    """build_problem for a synthetic case with some fields replaced (population / horizon / particles of a BASELINE config)."""
    import dataclasses

    import mbrl_lib_b200 as bp
    from mbrl_lib_b200 import functions

    spec = dataclasses.replace(syn.CASES[workload], **over)
    arrays = syn.make_model_arrays(spec)
    model = bp.model_from_arrays(spec, arrays, device)

    class _Env:
        observation_space = _Box(-np.inf, np.inf, spec.obs_dim)
        action_space = _Box(spec.action_lb, spec.action_ub, spec.act_dim)

    rew = functions.REWARD_FNS[spec.reward_fn] if spec.reward_fn else None
    env = bp.ModelEnv(_Env(), model, functions.TERM_FNS[spec.term_fn], rew,
                      generator=torch.Generator(device=device).manual_seed(0), precision="auto", ts1="tile_shuffle")
    return spec, arrays, env


def config3_icem_extra(device, flush, peak_tf):
    """BASELINE config 3: PETS Humanoid-v4 with iCEM (pop 1000, decay 1.3, coloured noise beta 2, keep 0.3, 5 iterations, H 40,
    20 particles; conf pets_icem_cartpole.yaml values) through ICEMOptimizer.optimize over evaluate_action_sequences.
    Two model shapes: the truncated-observation Humanoid (obs 45: inside the tensor-core plan) and the real Humanoid-v4
    dims (obs 376, in 393 -> out 754: outside it, served by the fp32 kernel).  Algorithmic FLOP per sequence = 2 sum K N x P x H."""
    import mbrl_lib_b200 as bp

    rows = []
    for name, reps in (("humanoid_trunc", 5), ("humanoid_v4", 2)):
        spec, _, env = build_problem_variant(device, name, population=1000, horizon=40, particles=20)
        H, A, P = spec.horizon, spec.act_dim, spec.particles
        lb, ub = np.full((H, A), spec.action_lb).tolist(), np.full((H, A), spec.action_ub).tolist()
        opt = bp.ICEMOptimizer(5, 0.1, 1000, 1.3, 2.0, lb, ub, 0.3, 0.1, device, return_mean_elites=True, population_size_module=5)
        obs0 = syn.make_rollout_inputs(spec, with_noise=False)["obs0"]
        seqs = {"n": 0}

        def obj(pop):
            seqs["n"] += pop.shape[0]
            return env.evaluate_action_sequences(pop, obs0, P)

        x0 = torch.zeros(H, A, device=device)
        opt.optimize(obj, x0=x0)
        torch.cuda.synchronize()
        seqs["n"] = 0
        ms = time_events(lambda: opt.optimize(obj, x0=x0), reps, flush)
        per_plan = seqs["n"] / reps
        dims = [(spec.in_size, spec.hid_size)] + [(spec.hid_size, spec.hid_size)] * (spec.num_layers - 1) + [(spec.hid_size, 2 * spec.out_size)]
        flop_seq = 2.0 * sum(k * n for k, n in dims) * P * H
        sps = per_plan / (ms * 1e-3)
        rows.append({"model": name, "obs_dim": spec.obs_dim, "in": spec.in_size, "out": 2 * spec.out_size, "kernel": env.precision,
                     "sequences_per_plan": per_plan, "ms_per_plan": ms, "sequences_per_s": sps,
                     "algorithmic_mflop_per_sequence": flop_seq / 1e6,
                     "tensor_roofline_frac": sps * flop_seq / 1e12 / peak_tf if env.precision == "bf16_tc" else None,
                     "tflops": sps * flop_seq / 1e12})
    return {"workload": "PETS Humanoid iCEM: pop 1000 decaying by 1.3, 5 iterations, H 40, 20 particles, coloured noise beta 2, "
                        "keep_elite_frac 0.3 (ICEMOptimizer.optimize over evaluate_action_sequences, CUDA events per plan)",
            "rows": rows}


def config4_mbpo_loop_extra(device):
    """BASELINE config 4 as MBPO runs it (mbrl/algorithms/mbpo.py:31-63): 100 000 start states x k model steps with an actor
    between the steps, transitions into a SAC buffer.  Device loop (mbpo.rollout_model_and_populate_sac_buffer: states,
    predictions and the accum_dones mask stay in HBM, one D2H of the compacted transitions) vs the reference-shaped numpy
    loop over ModelEnv.step (per-step H2D / D2H and host masking).  The actor is a fixed tanh-linear map (a torch callable on
    the device in the first case, numpy in the second)."""
    from mbrl_lib_b200 import mbpo

    spec, _, env = build_problem(device, "mbpo_halfcheetah")
    B, k = 100000, 5
    inp = syn.make_step_inputs(spec, B)
    W = torch.from_numpy(np.random.default_rng(0).standard_normal((spec.obs_dim, spec.act_dim)).astype(np.float32) * 0.3).to(device)
    Wh = W.cpu().numpy()

    class _Batch:
        def astuple(self):
            return (inp["obs"], None, None, None, None, None)

    class _Replay:
        def sample(self, n):
            return _Batch()

    class _Sac:
        rows = 0

        def add_batch(self, obs, action, next_obs, reward, terminated, truncated):
            _Sac.rows += len(obs)

    class _TorchAgent:
        def act_torch(self, obs, sample):
            return torch.tanh(obs @ W)

    class _NumpyAgent:
        def act(self, obs, sample=False, batched=False):
            return np.tanh(obs @ Wh).astype(np.float32)

    def device_loop():
        mbpo.rollout_model_and_populate_sac_buffer(env, _Replay(), _TorchAgent(), _Sac(), True, k, B)

    def numpy_loop():  # the reference's loop body over our ModelEnv.step (numpy in, numpy out, every step)
        agent = _NumpyAgent()
        sac = _Sac()
        model_state = env.reset(inp["obs"], return_as_np=True)
        accum = np.zeros(B, dtype=bool)
        obs = inp["obs"]
        for _ in range(k):
            action = agent.act(obs, sample=True, batched=True)
            pred_next, pred_rew, pred_done, model_state = env.step(action, model_state, sample=True)
            keep = ~accum
            sac.add_batch(obs[keep], action[keep], pred_next[keep], pred_rew[keep, 0], pred_done[keep, 0], np.zeros(keep.sum(), bool))
            obs = pred_next
            accum |= pred_done.squeeze()

    out = {}
    for name, fn in (("device_loop", device_loop), ("numpy_loop", numpy_loop)):
        fn()
        torch.cuda.synchronize()
        _Sac.rows = 0
        t0 = time.perf_counter()
        reps = 3
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / reps
        out[name + "_ms"] = dt * 1e3
        out[name + "_transitions_per_s"] = _Sac.rows / reps / dt
    out["workload"] = f"MBPO HalfCheetah model rollouts: {B} start states x {k} steps, actor between steps, transitions to a SAC buffer (host wall clock)"
    out["pcie_bytes_numpy_loop_per_step"] = B * ((spec.obs_dim + spec.act_dim) * 4 + (spec.obs_dim + 1) * 4 + 1)
    out["pcie_bytes_device_loop_total"] = B * spec.obs_dim * 4 + k * B * ((2 * spec.obs_dim + spec.act_dim + 1) * 4 + 1)
    return out


def run_ours(args):
    import torch.distributed as dist
    import mbrl_lib_b200 as bp
    from mbrl_lib_b200.planning import _FusedObjective

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = f"cuda:{local}"
    # the optimisers seed their sampling streams with torch.initial_seed(), which torch draws afresh in every process:
    # pin it so that a run's plans depend on its arguments only
    torch.manual_seed(0)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(device))
    spec, arrays, env = build_problem(device)
    inp = syn.make_rollout_inputs(spec, with_noise=False)
    H, A, N, P = spec.horizon, spec.act_dim, spec.population, spec.particles
    lb = np.full((H, A), spec.action_lb).tolist()
    ub = np.full((H, A), spec.action_ub).tolist()
    obs0 = inp["obs0"]
    x0 = torch.zeros(H, A, device=device)
    flush = l2_flush_buffer(device)
    seqs_per_step = CEM_ITERS * N * world
    warmup = max(args.warmup, 3)

    if world == 1:
        opt = bp.CEMOptimizer(CEM_ITERS, ELITE_RATIO, N, lb, ub, ALPHA, device, return_mean_elites=True)
        obj = _FusedObjective(env, obs0, P)

        def step():
            return opt.optimize(obj, x0=x0)
        if os.environ.get("B200PETS_CEM_MERGED", "1") == "0":
            launches_per_step = 1 + CEM_ITERS * 3  # init + (sample, rollout, refit incl. particle mean) per iteration
        else:  # init, first population, then per iteration: rollout + ONE refit-and-next-population kernel
            launches_per_step = 2 + CEM_ITERS * 2
    else:
        from mbrl_lib_b200.dist import ShardedCEMOptimizer

        opt = ShardedCEMOptimizer(CEM_ITERS, ELITE_RATIO, N * world, lb, ub, ALPHA, device, return_mean_elites=True)
        obj = _FusedObjective(env, obs0, P)

        def step():
            return opt.optimize(obj, x0=x0)
        if os.environ.get("B200PETS_PEER_EXCHANGE", "1") != "0":
            # first population, then per iteration: rollout, particle mean, values push, global select + elite push + refit + next population
            launches_per_step = 1 + CEM_ITERS * 4
        else:
            launches_per_step = CEM_ITERS * 5  # sample, rollout, particle mean, local top-k, refit-from-records (+ 1 NCCL kernel)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # ---- device-resident timing: per-step CUDA events, L2 flushed (untimed) between steps ----
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for s, e in evs:
        flush.fill_(1)
        s.record()
        out = step()
        e.record()
    barrier()
    step_ms = [s.elapsed_time(e) for s, e in evs]
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "solution.npy"), out.float().cpu().numpy())
    total_ms = torch.tensor([sum(step_ms)], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())

    # ---- dominant kernel (the rollout) alone, for the roofline ----
    pop = torch.from_numpy(inp["actions"]).to(device)
    for _ in range(3):
        env.evaluate_action_sequences(pop, obs0, P)
    torch.cuda.synchronize()
    kern_ms_avg = time_events(lambda: env.evaluate_action_sequences(pop, obs0, P), max(args.steps, 10), flush)

    # ---- end to end through the public API: agent.act(obs): H2D obs (pinned) ... D2H plan ----
    e2e = None
    if world == 1:
        cfg = {"_target_": "mbrl_lib_b200.TrajectoryOptimizerAgent", "planning_horizon": H, "replan_freq": 1, "verbose": False,
               "optimizer_cfg": {"_target_": "mbrl_lib_b200.CEMOptimizer", "num_iterations": CEM_ITERS,
                                 "elite_ratio": ELITE_RATIO, "population_size": N, "alpha": ALPHA, "device": device,
                                 "return_mean_elites": True}}
        agent = bp.create_trajectory_optim_agent_for_model(env, cfg, num_particles=P)
        for _ in range(3):
            agent.act(obs0)
        torch.cuda.synchronize()
        dt = 0.0
        for _ in range(args.steps):
            flush.fill_(1)
            torch.cuda.synchronize()  # the L2 flush is not part of the measured call
            t0 = time.perf_counter()
            a = agent.act(obs0)  # host numpy in (H2D from pinned memory), host numpy out (synchronises on the D2H of the plan)
            dt += time.perf_counter() - t0
        assert a.shape == (A,)
        e2e = {"value": CEM_ITERS * N * args.steps / dt, "unit": "sequences/s", "h2d_bytes_per_step": spec.obs_dim * 4,
               "d2h_bytes_per_step": H * A * 4, "ms_per_step": dt / args.steps * 1e3,
               "note": "agent.act(obs) per call, host wall clock; L2 flushed (untimed) before every call"}
    else:
        # sharded plan through the public API: host observation in (pinned H2D inside optimize), host plan out
        pin = torch.empty(H, A, dtype=torch.float32).pin_memory()
        for _ in range(2):
            pin.copy_(opt.optimize(obj, x0=x0), non_blocking=True)
            torch.cuda.synchronize()
        dt = 0.0
        for _ in range(args.steps):
            flush.fill_(1)
            barrier()
            t0 = time.perf_counter()
            pin.copy_(opt.optimize(obj, x0=x0), non_blocking=True)
            torch.cuda.synchronize()
            dt += time.perf_counter() - t0
        dt_t = torch.tensor([dt], device=device, dtype=torch.float64)
        dist.all_reduce(dt_t, op=dist.ReduceOp.MAX)
        dt = float(dt_t.item())
        e2e = {"value": seqs_per_step * args.steps / dt, "unit": "sequences/s", "h2d_bytes_per_step": spec.obs_dim * 4,
               "d2h_bytes_per_step": H * A * 4, "ms_per_step": dt / args.steps * 1e3,
               "note": "ShardedCEMOptimizer.optimize per call on every rank (max over ranks), host wall clock; L2 flushed before"}

    peak_tf, peak_src = measured_peak_tflops()
    extras = {}
    # ---- the exact-reference TS1 mode (explicit torch.randperm per step, one launch per step), for comparison ----
    if world == 1 and not args.no_scan:
        _, _, env_perm = build_problem(device, ts1="perms")
        B = N * P
        perms = torch.stack([torch.randperm(B, device=device) for _ in range(H)])
        for _ in range(2):
            env_perm.evaluate_action_sequences(pop, obs0, P, _perms=perms)
        ms_inj = time_events(lambda: env_perm.evaluate_action_sequences(pop, obs0, P, _perms=perms), 10, flush)
        ms_gen = time_events(lambda: env_perm.evaluate_action_sequences(pop, obs0, P), 10, flush)
        extras["ts1_perms_mode"] = {
            "what": "evaluate_action_sequences of 500 sequences with ts1='perms': the reference's per-step randperm of all "
                    "10 000 rows (gaussian_mlp.py:202-212), one kernel launch per horizon step, row state through HBM",
            "ms_permutations_given": ms_inj, "sequences_per_s_permutations_given": N / (ms_inj * 1e-3),
            "ms_with_torch_randperm": ms_gen, "sequences_per_s_with_torch_randperm": N / (ms_gen * 1e-3),
            "tile_shuffle_ms": kern_ms_avg}
    # ---- population scan of the rollout alone (BASELINE.json config 5 shape, one GPU): fills all SMs ----
    if world == 1 and not args.no_scan:
        scan = []
        for scale in (2, 8, 32, 128):
            big = pop.repeat(scale, 1, 1)
            for _ in range(2):
                env.evaluate_action_sequences(big, obs0, P)
            torch.cuda.synchronize()
            ms = time_events(lambda: env.evaluate_action_sequences(big, obs0, P), 5)
            sps = big.shape[0] / (ms * 1e-3)
            scan.append({"population": int(big.shape[0]), "ms": ms, "sequences_per_s": sps,
                         "tensor_roofline_frac": sps * FLOP_PER_SEQ / 1e12 / peak_tf})
            del big
        extras["population_scan_rollout_only"] = scan
        extras["config4_mbpo_step"] = mbpo_step_extra(device, flush)
        for key, fn in (("config3_humanoid_icem", lambda: config3_icem_extra(device, flush, peak_tf)),
                        ("config4_mbpo_rollout_loop", lambda: config4_mbpo_loop_extra(device))):
            try:  # extra lines must never take the headline measurement down with them
                extras[key] = fn()
            except Exception as exc:  # pragma: no cover - depends on the box
                extras[key] = {"error": f"{type(exc).__name__}: {exc}"}
    # ---- config 5: fixed GLOBAL population sharded over the ranks (strong scaling), collective share of an iteration ----
    if world > 1 and not args.no_scan5:
        from mbrl_lib_b200.dist import ShardedCEMOptimizer

        scan5 = []
        for gpop in (8000, 16000, 64000):
            o5 = ShardedCEMOptimizer(CEM_ITERS, ELITE_RATIO, gpop, lb, ub, ALPHA, device, return_mean_elites=True)
            for _ in range(2):
                o5.optimize(obj, x0=x0)
            barrier()
            o5.comm_events = []
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 3
            barrier()
            s.record()
            for _ in range(reps):
                o5.optimize(obj, x0=x0)
            e.record()
            barrier()
            ms = torch.tensor([s.elapsed_time(e) / reps], device=device, dtype=torch.float64)
            comm = torch.tensor([sum(a.elapsed_time(b) for a, b in o5.comm_events) / reps], device=device, dtype=torch.float64)
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(comm, op=dist.ReduceOp.MAX)
            o5.comm_events = None
            scan5.append({"global_population": gpop, "ms_per_plan": float(ms), "sequences_per_s": CEM_ITERS * gpop / (float(ms) * 1e-3),
                          "collective_ms_per_plan": float(comm), "collective_share": float(comm) / float(ms),
                          "tensor_roofline_frac_per_gpu": CEM_ITERS * gpop / (float(ms) * 1e-3) * FLOP_PER_SEQ / 1e12 / peak_tf / world})
            del o5
        extras["config5_population_scan_sharded"] = {
            "what": "full 5-iteration plan, global population fixed and sharded over the ranks (strong scaling in N); "
                    "collective = the exchange of the iteration, timed with CUDA events around it (includes waiting for the slowest "
                    "rank): peer-memory path = values push + global select + elite push + refit + next population (two kernels); "
                    "B200PETS_PEER_EXCHANGE=0 = NCCL all-gather of local top-k records only", "rows": scan5}
    clocks = sampler.stop() if rank == 0 else None

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baseline(spec, arrays, reps=3)

    if rank == 0:
        achieved = N * FLOP_PER_SEQ / (kern_ms_avg * 1e-3) / 1e12
        traffic, traffic_src = ncu_dram_traffic()
        line = {
            "metric": METRIC, "value": seqs_per_step * args.steps / (total_ms * 1e-3), "unit": "sequences/s",
            "n_gpus": world, "steps": args.steps, "warmup": warmup, "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if env.precision == "bf16_tc" else "f32",
            "data": "synthetic", "config": dict(CONFIG),
            "impl_notes": {"ts1": "in-kernel tile shuffle (member per shuffle group and step from Philox; exact-oracle parity in "
                                  "tests/test_gpu_shuffle.py)", "population_per_gpu": N, "sequences_per_step": seqs_per_step,
                           "parallelism": f"population-sharded x{world}",
                           "l2": "flushed between timed steps (256 MB write, untimed); weights (1.3 MB) are re-fetched every step",
                           "precision": env.precision},
            "gpu_launches": launches_per_step * args.steps,
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                         "traffic": traffic, "traffic_source": f"ncu --set full dram__bytes_read.sum + dram__bytes_write.sum of one launch ({traffic_src}); "
                         "algorithmic: 1.3 MB bf16 weights + 0.36 MB actions + 2 KB returns",
                         "kernel": "rollout_tc_kernel (one CEM iteration: 500 sequences x 20 particles x 30 steps)",
                         "kernel_ms": kern_ms_avg, "peak_source": peak_src, "algorithmic_flop_per_launch": N * FLOP_PER_SEQ},
            "clocks": clocks,
        }
        if e2e:
            line["e2e"] = e2e
        if cpu:
            line["cpu_baseline"] = cpu
        line.update(extras)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------------
# CPU legs
# ------------------------------------------------------------------------------------------------------------------
def _reference_objects(spec, arrays):
    """(kind, evaluate(actions) callable, act(obs) callable or None, source)."""
    from baseline import reference_arm as ra

    mbrl, src = ra.import_reference()
    if mbrl is not None:
        env = ra.build_model_env(mbrl, spec, arrays)
        agent = ra.build_agent(mbrl, env, spec, CEM_ITERS, ELITE_RATIO, ALPHA)
        obs0 = syn.make_rollout_inputs(spec, with_noise=False)["obs0"]
        return ("reference", lambda acts: env.evaluate_action_sequences(acts, obs0, spec.particles), agent.act,
                os.path.relpath(src, ROOT) if src.startswith(ROOT) else src)
    from oracle import pets_oracle as po

    model = po.OracleModel(spec, arrays)
    obs0 = syn.make_rollout_inputs(spec, with_noise=False)["obs0"]
    gen = torch.Generator().manual_seed(0)

    def evaluate(acts):  # the RNG work the reference does per step stays inside the timed region
        Hh, B = spec.horizon, acts.shape[0] * spec.particles
        perms = torch.stack([torch.randperm(B, generator=gen) for _ in range(Hh)])
        eps = torch.randn(Hh, B, spec.out_size, generator=gen)
        return model.evaluate_action_sequences(acts, obs0, spec.particles, perms, eps)

    return "port", evaluate, None, f"oracle port ({src})"


def pick_cpu_threads(evaluate, actions):
    """torch's default (one thread per hardware thread) oversubscribes these small GEMMs badly on a many-core host;
    time a 50-sequence slice at a few thread counts and keep the fastest."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu})
    small = actions[:50]
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        evaluate(small)
        t0 = time.perf_counter()
        evaluate(small)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def cpu_baseline(spec, arrays, reps=3):
    kind, evaluate, _, src = _reference_objects(spec, arrays)
    actions = torch.from_numpy(syn.make_rollout_inputs(spec, with_noise=False)["actions"])
    threads = pick_cpu_threads(evaluate, actions)
    evaluate(actions)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        evaluate(actions)
        ts.append(time.perf_counter() - t0)
    med = statistics.median(ts)
    what = ("the reference's own ModelEnv.evaluate_action_sequences (mbrl-lib from " + src + ")") if kind == "reference" else \
        "oracle port of the reference's fp32 PyTorch path"
    return {"value": spec.population / med, "unit": "sequences/s", "cores": threads, "kind": kind,
            "sample": f"{reps} x evaluate_action_sequences of 500 sequences (one CEM iteration), {what}, "
                      f"best of thread counts up to {os.cpu_count()}, median {med:.3f} s"}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path on the host cores (rank 0 only).
    One step = one TrajectoryOptimizerAgent.act() = one 5-iteration CEM plan (2 500 sequences), as on our arm."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    spec = syn.CASES[WORKLOAD]
    arrays = syn.make_model_arrays(spec)
    kind, evaluate, act, src = _reference_objects(spec, arrays)
    inp = syn.make_rollout_inputs(spec, with_noise=False)
    actions = torch.from_numpy(inp["actions"])
    cores = pick_cpu_threads(evaluate, actions)
    if act is None:  # oracle port: five evaluations stand in for a plan (sampler / refit are negligible on the CPU)
        def act(_obs):
            for _ in range(CEM_ITERS):
                evaluate(actions)
    steps, warmup = args.steps, max(args.warmup, 1)
    for _ in range(warmup):
        act(inp["obs0"])
    t0 = time.perf_counter()
    for _ in range(steps):
        act(inp["obs0"])
    dt = time.perf_counter() - t0
    val = CEM_ITERS * spec.population * steps / dt
    sample = (f"{steps} x agent.act() (5 CEM iterations x 500 sequences each) of the "
              f"{'unmodified reference (' + src + ')' if kind == 'reference' else 'oracle port'}, torch CPU fp32, {cores} threads "
              f"(fastest of the thread counts tried on {os.cpu_count()} hardware threads)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "sequences/s", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
        "steps": steps, "warmup": warmup, "ms_per_step": dt / steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": dict(CONFIG),
        "impl_notes": {"ts1": "torch.randperm per step (the reference's rule)", "device": "cpu", "source": src},
        "cpu_baseline": {"value": val, "unit": "sequences/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "sequences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--no-scan5", action="store_true", help="skip the sharded config-5 population scan (N > 1)")
    ap.add_argument("--no-scan", action="store_true", help="skip the population scan / extra configurations")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's plan to DIR/solution.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the plan of the CUDA path; the reference arm draws its own random streams, "
                 "so its outputs are not comparable output for output")
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
