"""Generate golden vectors from the *imported reference* (mbrl-lib at /root/reference) -- run in the build
container only:

    PYTHONPATH=oracle/ref_shims:/root/reference python oracle/gen_golden.py

The reference's RNG calls (torch.randperm, torch.normal, truncated_normal_) are monkey-fed the same
injected draws that `mbrl_lib_b200.synthetic` regenerates from numpy seeds anywhere, so the committed
`tests/golden/*.npz` hold only outputs + input checksums.  TEST INFRASTRUCTURE; nothing shipped uses it.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mbrl.env.reward_fns as ref_rew  # noqa: E402
import mbrl.env.termination_fns as ref_term  # noqa: E402
import mbrl.models  # noqa: E402
import mbrl.planning  # noqa: E402
import mbrl.util.math  # noqa: E402

from mbrl_lib_b200 import synthetic as syn  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
ACT = {"relu": "torch.nn.ReLU", "silu": "torch.nn.SiLU", "leaky_relu": "torch.nn.LeakyReLU"}


def _proc_fn(name):
    if name is None:
        return None
    if name == "halfcheetah":  # mbrl/env/pets_halfcheetah.py:91-113 (module needs mujoco to import)
        return lambda s: torch.cat([s[..., 1:2], torch.sin(s[..., 2:3]), torch.cos(s[..., 2:3]), s[..., 3:]], dim=-1)
    if name == "cartpole":  # mbrl/env/pets_cartpole.py:78-101
        return lambda s: torch.cat([torch.sin(s[..., 1:2]), torch.cos(s[..., 1:2]), s[..., :1], s[..., 2:]], dim=-1)
    raise ValueError(name)


class _Env:
    def __init__(self, spec):
        import gymnasium

        self.observation_space = gymnasium.spaces.Box(-np.inf, np.inf, (spec.obs_dim,))
        self.action_space = gymnasium.spaces.Box(spec.action_lb, spec.action_ub, (spec.act_dim,))


def build_reference(spec, arrays):
    """Reference GaussianMLP + OneDTransitionRewardModel + ModelEnv carrying the synthetic weights."""
    model = mbrl.models.GaussianMLP(
        spec.in_size, spec.out_size, "cpu", num_layers=spec.num_layers, ensemble_size=spec.ensemble_size,
        hid_size=spec.hid_size, deterministic=spec.deterministic, propagation_method=spec.propagation,
        activation_fn_cfg={"_target_": ACT[spec.activation]})
    with torch.no_grad():
        for li, layer in enumerate(model.hidden_layers):
            layer[0].weight.copy_(torch.from_numpy(arrays["weights"][li]))
            layer[0].bias.copy_(torch.from_numpy(arrays["biases"][li]))
        model.mean_and_logvar.weight.copy_(torch.from_numpy(arrays["weights"][-1]))
        model.mean_and_logvar.bias.copy_(torch.from_numpy(arrays["biases"][-1]))
        if not spec.deterministic:
            model.min_logvar.copy_(torch.from_numpy(arrays["min_logvar"]))
            model.max_logvar.copy_(torch.from_numpy(arrays["max_logvar"]))
    wrapper = mbrl.models.OneDTransitionRewardModel(
        model, target_is_delta=spec.target_is_delta, normalize=spec.normalize is not None,
        normalize_double_precision=spec.normalize == "float64", learned_rewards=spec.learned_rewards,
        obs_process_fn=_proc_fn(spec.obs_process), no_delta_list=list(spec.no_delta_list),
        num_elites=spec.num_models)
    if spec.normalize is not None:
        wrapper.input_normalizer.mean = torch.from_numpy(arrays["norm_mean"])
        wrapper.input_normalizer.std = torch.from_numpy(arrays["norm_std"])
    if spec.elites is not None:
        wrapper.set_elite(list(spec.elites))
    reward_fn = getattr(ref_rew, spec.reward_fn) if spec.reward_fn else None
    term_fn = getattr(ref_term, spec.term_fn)
    env = mbrl.models.ModelEnv(_Env(spec), wrapper, term_fn, reward_fn, generator=torch.Generator())
    return env


class FeedRNG:
    """Context manager: torch.randperm / torch.normal / truncated_normal_ return injected draws in call order."""

    def __init__(self, perms=(), normals=(), truncs=()):
        self.perms, self.normals, self.truncs = list(perms), list(normals), list(truncs)

    def __enter__(self):
        self._rp, self._nm, self._tn = torch.randperm, torch.normal, mbrl.util.math.truncated_normal_

        def randperm(n, **kw):
            p = self.perms.pop(0)
            assert p.numel() == n, (p.numel(), n)
            return p

        def normal(mean, std, *a, **kw):
            z = self.normals.pop(0)
            assert z.shape == mean.shape, (z.shape, mean.shape)
            return mean + std * z

        def trunc(tensor, mean=0, std=1):
            z = self.truncs.pop(0)
            tensor.copy_(z * std + mean)
            return tensor

        torch.randperm, torch.normal, mbrl.util.math.truncated_normal_ = randperm, normal, trunc
        return self

    def __exit__(self, *a):
        torch.randperm, torch.normal, mbrl.util.math.truncated_normal_ = self._rp, self._nm, self._tn
        assert not self.perms and not self.truncs, "unused injected draws"


def gen_rollout(name):
    spec = syn.CASES[name]
    arrays = syn.make_model_arrays(spec)
    inp = syn.make_rollout_inputs(spec)
    env = build_reference(spec, arrays)
    H = spec.horizon
    perms = [torch.from_numpy(p) for p in inp["perms"]]
    if spec.propagation == "expectation":
        perms = []
    normals = [] if spec.deterministic else [torch.from_numpy(inp["eps"][t]) for t in range(H)]
    with FeedRNG(perms=perms, normals=normals):
        ret = env.evaluate_action_sequences(torch.from_numpy(inp["actions"]), inp["obs0"], spec.particles)
    np.savez(os.path.join(GOLD, f"rollout_{name}.npz"), returns=ret.numpy(),
             model_sum=syn.checksum(arrays), input_sum=syn.checksum(inp))
    print(name, "returns", ret[:4].tolist())


def gen_step(name, batch):
    spec = syn.CASES[name]
    arrays = syn.make_model_arrays(spec)
    inp = syn.make_step_inputs(spec, batch)
    env = build_reference(spec, arrays)
    with FeedRNG(perms=[torch.from_numpy(inp["perm"])], normals=[torch.from_numpy(inp["eps"])]):
        # ModelEnv.reset draws the TSinf permutation if the model is fixed_model
        if spec.propagation == "fixed_model":
            st = env.reset(inp["obs"], return_as_np=True)
        else:
            st = env.reset(inp["obs"], return_as_np=True)
        nobs, rew, done, _ = env.step(inp["act"], st, sample=True)
    np.savez(os.path.join(GOLD, f"step_{name}.npz"), next_obs=nobs, reward=rew, done=done,
             model_sum=syn.checksum(arrays), input_sum=syn.checksum(inp))
    print("step", name, nobs[0, :3], rew[0], done.sum())


def quad_objective(target):
    def f(pop):
        return -((pop - target) ** 2).sum(dim=(1, 2)) + 0.3 * torch.sin(3.0 * pop).sum(dim=(1, 2))

    return f


def gen_cem(tag, clipped, return_mean):
    g = np.random.default_rng(1234 + clipped)
    N, H, A, iters = 64, 5, 3, 4
    lb = torch.tensor(np.tile([-1.0, -0.5, -2.0], (H, 1)), dtype=torch.float32)
    ub = torch.tensor(np.tile([1.0, 0.5, 2.0], (H, 1)), dtype=torch.float32)
    z = g.standard_normal((iters, N, H, A)).astype(np.float32)
    if not clipped:
        z = np.clip(z, -2, 2)  # any values in [-2, 2] are valid truncated-normal draws
    target = torch.tensor(g.uniform(-0.4, 0.4, (H, A)).astype(np.float32))
    x0 = torch.tensor(g.uniform(-0.2, 0.2, (H, A)).astype(np.float32))
    opt = mbrl.planning.CEMOptimizer(iters, 0.15, N, lb.tolist(), ub.tolist(), 0.1, "cpu",
                                     return_mean_elites=return_mean, clipped_normal=clipped)
    trace = []

    def cb(pop, vals, i):
        trace.append((pop.clone(), vals.clone()))

    feed = dict(normals=[torch.from_numpy(z[i]) for i in range(iters)]) if clipped else \
        dict(truncs=[torch.from_numpy(z[i]) for i in range(iters)])
    if clipped:
        rl = torch.randn_like

        def randn_like(t, **kw):
            return feed["normals"].pop(0)

        torch.randn_like = randn_like
        try:
            sol = opt.optimize(quad_objective(target), x0=x0, callback=cb)
        finally:
            torch.randn_like = rl
    else:
        with FeedRNG(**feed):
            sol = opt.optimize(quad_objective(target), x0=x0, callback=cb)
    np.savez(os.path.join(GOLD, f"cem_{tag}.npz"), z=z, lb=lb.numpy(), ub=ub.numpy(), target=target.numpy(),
             x0=x0.numpy(), solution=sol.numpy(), pops=np.stack([t[0].numpy() for t in trace]),
             values=np.stack([t[1].numpy() for t in trace]), iters=iters, N=N, elite_ratio=0.15, alpha=0.1)
    print("cem", tag, sol[0].tolist())


def gen_icem():
    g = np.random.default_rng(77)
    H, A, iters, pop0 = 8, 2, 4, 48
    elite_ratio, decay, beta, keep_frac, alpha, module = 0.125, 1.3, 2.0, 0.5, 0.1, 3
    lb = torch.tensor(np.tile([-1.0, -0.5], (H, 1)), dtype=torch.float32)
    ub = torch.tensor(np.tile([1.0, 0.5], (H, 1)), dtype=torch.float32)
    target = torch.tensor(g.uniform(-0.4, 0.4, (H, A)).astype(np.float32))
    x0 = torch.tensor(g.uniform(-0.2, 0.2, (H, A)).astype(np.float32))
    opt = mbrl.planning.ICEMOptimizer(iters, elite_ratio, pop0, decay, beta, lb.tolist(), ub.tolist(), keep_frac,
                                      alpha, "cpu", return_mean_elites=False, population_size_module=module)
    elite_num, keep = int(opt.elite_num), int(opt.keep_elite_size)
    sizes = []
    for i in range(iters):
        n = int(np.ceil(max(pop0 * decay ** -i, 2 * elite_num)))
        n = n if n % module == 0 else n + module - n % module
        sizes.append(n)
    out = {"sizes": np.array(sizes), "keep": keep, "elite_num": elite_num}
    sols = []
    for call in range(2):  # second call exercises the kept/shifted elites of iteration 0
        normals, perms = [], []
        rec = {}
        for i in range(iters):
            sr = g.standard_normal((sizes[i], A, H // 2 + 1)).astype(np.float32)
            si = g.standard_normal((sizes[i], A, H // 2 + 1)).astype(np.float32)
            normals += [torch.from_numpy(sr), torch.from_numpy(si)]
            rec[f"sr{i}"], rec[f"si{i}"] = sr, si
            if call > 0 or i > 0:
                p = g.permutation(elite_num).astype(np.int64)
                perms.append(torch.from_numpy(p))
                rec[f"perm{i}"] = p
                if i == 0:
                    e = g.standard_normal((keep, A)).astype(np.float32)
                    normals.append(torch.from_numpy(e))
                    rec["end_eps"] = e
        trace = []
        with FeedRNG(perms=perms, normals=normals):
            sol = opt.optimize(quad_objective(target), x0=x0, callback=lambda p, v, i: trace.append((p.clone(), v.clone())))
        sols.append(sol.numpy())
        for k, v in rec.items():
            out[f"c{call}_{k}"] = v
        for i, (p, v) in enumerate(trace):
            out[f"c{call}_pop{i}"] = p.numpy()
            out[f"c{call}_val{i}"] = v.numpy()
        out[f"c{call}_elite"] = opt.elite.numpy()
    np.savez(os.path.join(GOLD, "icem.npz"), lb=lb.numpy(), ub=ub.numpy(), target=target.numpy(), x0=x0.numpy(),
             sol0=sols[0], sol1=sols[1], iters=iters, pop0=pop0, elite_ratio=elite_ratio, decay=decay, beta=beta,
             keep_frac=keep_frac, alpha=alpha, module=module, **out)
    print("icem", sols[1][0].tolist())


def gen_mppi():
    g = np.random.default_rng(99)
    N, H, A, iters = 48, 6, 2, 3
    lb = torch.tensor(np.tile([-1.0, -0.5], (H, 1)), dtype=torch.float32)
    ub = torch.tensor(np.tile([1.0, 0.5], (H, 1)), dtype=torch.float32)
    target = torch.tensor(g.uniform(-0.4, 0.4, (H, A)).astype(np.float32))
    opt = mbrl.planning.MPPIOptimizer(iters, N, 0.9, 0.5, 0.7, lb.tolist(), ub.tolist(), "cpu")
    out = {}
    for call in range(2):
        z = np.clip(g.standard_normal((iters, N, H, A)), -2, 2).astype(np.float32)
        trace = []
        with FeedRNG(truncs=[torch.from_numpy(z[k]) for k in range(iters)]):
            sol = opt.optimize(quad_objective(target), callback=lambda p, v, k: trace.append((p.clone(), v.clone())))
        out[f"z{call}"] = z
        out[f"sol{call}"] = sol.numpy()
        out[f"pops{call}"] = np.stack([t[0].numpy() for t in trace])
    np.savez(os.path.join(GOLD, "mppi.npz"), lb=lb.numpy(), ub=ub.numpy(), target=target.numpy(), iters=iters, N=N,
             gamma=0.9, sigma=0.5, beta=0.7, **out)
    print("mppi", out["sol1"][0].tolist())


def gen_cem_model():
    """Full CEM over the model rollout (small halfcheetah case): pins optimiser+rollout composition."""
    spec = syn.CASES["halfcheetah_small"]
    arrays = syn.make_model_arrays(spec)
    inp = syn.make_rollout_inputs(spec)
    env = build_reference(spec, arrays)
    N, H, A, P, iters = spec.population, spec.horizon, spec.act_dim, spec.particles, 3
    nz = syn.make_cem_noise(spec, iters)
    z, eps, perms = nz["z"], nz["eps"], nz["perms"]
    lb = np.tile(np.full(A, spec.action_lb), (H, 1)).tolist()
    ub = np.tile(np.full(A, spec.action_ub), (H, 1)).tolist()
    opt = mbrl.planning.CEMOptimizer(iters, 0.1, N, lb, ub, 0.1, "cpu", return_mean_elites=True)
    vals = []
    feed = FeedRNG(perms=[torch.from_numpy(perms[i, t]) for i in range(iters) for t in range(H)],
                   normals=[torch.from_numpy(eps[i, t]) for i in range(iters) for t in range(H)],
                   truncs=[torch.from_numpy(z[i]) for i in range(iters)])
    with feed:
        sol = opt.optimize(lambda pop: env.evaluate_action_sequences(pop, inp["obs0"], P),
                           x0=torch.zeros(H, A), callback=lambda p, v, i: vals.append(v.clone().numpy()))
    np.savez(os.path.join(GOLD, "cem_model.npz"), noise_sum=syn.checksum(nz), solution=sol.numpy(),
             values=np.stack(vals), iters=iters)
    print("cem_model", sol[0].tolist())


def gen_counter_world():
    """The reference's closed-form case (tests/core/test_models.py:365-385) run through the REAL GaussianMLP path
    with the hand-built ReLU ensemble of synthetic.counter_world: returns must be H(H+1)/2 * a exactly."""
    spec, arrays = syn.counter_world()
    env = build_reference(spec, arrays)
    N = 4
    grid = np.zeros((9, 9, 2), np.float32)
    for P in range(1, 10):
        for H in range(1, 10):
            for ai, a in enumerate((1.0, 2.0)):
                ret = env.evaluate_action_sequences(torch.full((N, H, 1), a), np.zeros(1), P)
                assert torch.equal(ret, torch.full((N,), H * (H + 1) / 2 * a)), (P, H, a, ret)
                grid[P - 1, H - 1, ai] = ret[0].item()
    np.savez(os.path.join(GOLD, "kat_counter_world.npz"), returns=grid, model_sum=syn.checksum(arrays))
    print("counter_world", grid[8, 8].tolist())


REFERENCE_OBJECT_CASES = ["halfcheetah_small", "cartpole", "hopper_tsinf", "pets_halfcheetah_small", "ant_learned_fn"]


def gen_reference_objects():
    """What tests/test_reference_objects.py checks the duck-typed boundary against: the recorded surface
    (oracle/ref_surface.py) of the reference's OneDTransitionRewardModel(GaussianMLP) per case, of its reward /
    termination callables, the shipped conf/action_optimizer/*.yaml and the optimizers' constructor arguments."""
    import inspect
    import json

    import yaml

    from oracle import ref_surface

    models = {}
    for name in REFERENCE_OBJECT_CASES:
        spec = syn.CASES[name]
        models[name] = ref_surface.record(build_reference(spec, syn.make_model_arrays(spec)).dynamics_model)
    # the drop-in object of tests/test_host_cpu.py: fp64 normaliser, reward from reward_fns, no learned rewards
    mlp = mbrl.models.GaussianMLP(23, 17, "cpu", num_layers=4, ensemble_size=7, hid_size=200,
                                  propagation_method="random_model", activation_fn_cfg={"_target_": "torch.nn.SiLU"})
    wrapper = mbrl.models.OneDTransitionRewardModel(mlp, target_is_delta=True, normalize=True,
                                                    normalize_double_precision=True, learned_rewards=False, num_elites=5)
    wrapper.set_elite([0, 2, 3, 5, 6])
    models["silu_fp64_normalizer"] = ref_surface.record(wrapper)
    conf = os.path.join(os.path.dirname(mbrl.__file__), "examples", "conf", "action_optimizer")
    yamls = {}
    for name in ("cem", "icem", "mppi"):
        with open(os.path.join(conf, f"{name}.yaml")) as f:
            yamls[name] = yaml.safe_load(f)
    ctor = {c: sorted(set(inspect.signature(getattr(mbrl.planning, c).__init__).parameters) - {"self"})
            for c in ("CEMOptimizer", "ICEMOptimizer", "MPPIOptimizer")}
    out = {"models": models,
           "reward_fns": {n: ref_surface.record(getattr(ref_rew, n))
                          for n in ("cartpole", "cartpole_pets", "inverted_pendulum", "halfcheetah", "pusher")},
           "termination_fns": {n: ref_surface.record(getattr(ref_term, n)) for n in
                               ("hopper", "cartpole", "inverted_pendulum", "no_termination", "walker2d", "ant", "humanoid")},
           "optimizer_yaml": yamls, "optimizer_ctor_args": ctor}
    with open(os.path.join(GOLD, "reference_objects.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("reference_objects", sorted(models))


if __name__ == "__main__":
    torch.manual_seed(0)
    os.makedirs(GOLD, exist_ok=True)
    for nm in ["cartpole", "halfcheetah", "halfcheetah_small", "pets_halfcheetah_small", "humanoid_trunc",
               "relu_expectation", "silu_expectation", "hopper_tsinf", "cartpole_pets", "pusher_det", "walker_ant", "humanoid_v4", "tc_hid64", "tc_wide", "tc_shallow", "ant_learned_fn"]:
        gen_rollout(nm)
    gen_step("mbpo_halfcheetah_small", 1000)
    gen_step("cartpole", 500)
    gen_cem("trunc_best", clipped=False, return_mean=False)
    gen_cem("trunc_mean", clipped=False, return_mean=True)
    gen_cem("clipped_best", clipped=True, return_mean=False)
    gen_icem()
    gen_mppi()
    gen_cem_model()
    gen_counter_world()
    gen_reference_objects()
