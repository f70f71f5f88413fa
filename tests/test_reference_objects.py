"""The drop-in boundary against REAL mbrl-lib objects (SURVEY.md 8b; VERDICT r1 "boundary is a mirror, never a plug-in").

``tests/golden/reference_objects.json`` holds what ``oracle/gen_golden.py`` recorded from the unmodified reference
(imported with the four absent pure-Python deps shimmed, ``oracle/ref_shims``): the attribute surface of its
``OneDTransitionRewardModel(GaussianMLP)`` objects, its reward / termination callables, the shipped
``conf/action_optimizer/{cem,icem,mppi}.yaml`` and the optimizers' constructor arguments.  ``oracle.ref_surface.rebuild``
turns a recorded model back into an object with exactly the recorded attributes, so the checks below read what
the real object exposes without mbrl-lib being installed:

* CPU: ``staging.StagedModel(stage=False)`` reads the recorded objects exactly as the kernels need them, the
  reference's own reward / termination callables resolve to device functions, and the shipped YAMLs instantiate
  through ``_instantiate`` into the B200 classes.
* GPU: OUR ``ModelEnv`` over the recorded reference object (weights filled in) must reproduce what the REFERENCE's
  ``ModelEnv.evaluate_action_sequences`` computed with the same injected draws (``tests/golden/rollout_<case>.npz``).

Three tests exercise mbrl-lib's own code (its trainer, normaliser and class hierarchy).  They import the unmodified
package that ``build()`` copies into ``oracle/_ref`` (``oracle/ref_install.py``) and skip where no copy could be made.
"""
import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from baseline import reference_arm as ra  # noqa: E402
from mbrl_lib_b200 import _lib, functions, staging, synthetic as syn  # noqa: E402
from oracle import ref_surface  # noqa: E402

mbrl, REF_SRC = ra.import_reference()
needs_ref = pytest.mark.skipif(mbrl is None, reason=f"mbrl-lib not importable here: {REF_SRC}")
with open(os.path.join(ROOT, "tests", "golden", "reference_objects.json")) as _f:
    RECORDED = json.load(_f)


def _recorded_model(name, device="cpu"):
    """The reference's OneDTransitionRewardModel(GaussianMLP) of case ``name`` as recorded, carrying the synthetic
    weights of the case (what oracle/gen_golden.py:build_reference loads into the real object)."""
    spec = syn.CASES[name]
    arrays = syn.make_model_arrays(spec)
    wrapper = ref_surface.rebuild(RECORDED["models"][name], device)
    mlp = wrapper.model
    for li, layer in enumerate(mlp.hidden_layers):
        layer[0].weight.copy_(torch.from_numpy(arrays["weights"][li]))
        layer[0].bias.copy_(torch.from_numpy(arrays["biases"][li]))
    mlp.mean_and_logvar.weight.copy_(torch.from_numpy(arrays["weights"][-1]))
    mlp.mean_and_logvar.bias.copy_(torch.from_numpy(arrays["biases"][-1]))
    if not spec.deterministic:
        mlp.min_logvar.copy_(torch.from_numpy(arrays["min_logvar"]))
        mlp.max_logvar.copy_(torch.from_numpy(arrays["max_logvar"]))
    if spec.normalize is not None:
        wrapper.input_normalizer.mean = torch.from_numpy(arrays["norm_mean"]).to(device)
        wrapper.input_normalizer.std = torch.from_numpy(arrays["norm_std"]).to(device)
    fn = wrapper.obs_process_fn
    if fn is not None:  # the reference's Env.preprocess_fn was restated as a lambda (the env modules need mujoco): tag it
        fn.b200pets_kind, fn.b200pets_name = "proc", spec.obs_process
    return spec, arrays, wrapper


def _recorded_callables(spec):
    """The reference's own reward_fns.<name> / termination_fns.<name> of the case (recorded module and name)."""
    rew = ref_surface.rebuild(RECORDED["reward_fns"][spec.reward_fn]) if spec.reward_fn else None
    return rew, ref_surface.rebuild(RECORDED["termination_fns"][spec.term_fn])


def _real_model(name="halfcheetah_small", device="cpu"):
    spec = syn.CASES[name]
    arrays = syn.make_model_arrays(spec)
    env = ra.build_model_env(mbrl, spec, arrays)
    fn = env.dynamics_model.obs_process_fn
    if fn is not None:  # reference_arm restates Env.preprocess_fn as a lambda (the env modules need mujoco): tag it
        fn.b200pets_kind, fn.b200pets_name = "proc", spec.obs_process
    if device != "cpu":
        env.dynamics_model.to(device)
        env.dynamics_model.device = torch.device(device)
        env.dynamics_model.model.device = torch.device(device)
        env.device = torch.device(device)
        nz = env.dynamics_model.input_normalizer
        if nz is not None:
            nz.mean, nz.std, nz.device = nz.mean.to(device), nz.std.to(device), torch.device(device)
        env._rng = torch.Generator(device=device)
    return spec, arrays, env


def test_staging_reads_a_real_reference_model():
    rec = RECORDED["models"]["halfcheetah_small"]  # recorded from mbrl-lib's own classes
    assert rec["class_module"].startswith("mbrl.models") and rec["attrs"]["model"]["class_module"].startswith("mbrl.models")
    assert (rec["class"], rec["attrs"]["model"]["class"]) == ("OneDTransitionRewardModel", "GaussianMLP")
    spec, arrays, wrapper = _recorded_model("halfcheetah_small")
    sm = staging.StagedModel(wrapper, *_recorded_callables(spec), stage=False)
    d = sm._describe()
    assert (d.ensemble_size, d.num_members) == (spec.ensemble_size, spec.num_models)
    assert (d.in_size, d.out_size, d.hid_size, d.num_hidden) == (spec.in_size, spec.out_size, spec.hid_size, spec.num_layers)
    assert (d.obs_dim, d.act_dim) == (spec.obs_dim, spec.act_dim)
    assert d.activation == _lib.ACT[spec.activation]
    assert d.norm_mode == {None: 0, "float32": 1, "float64": 2}[spec.normalize]
    assert d.learned_rewards == int(spec.learned_rewards) and d.target_is_delta == int(spec.target_is_delta)
    assert d.reward_fn == _lib.REWARD[spec.reward_fn] and d.term_fn == _lib.TERM[spec.term_fn]
    assert sm.members() == list(spec.elites)  # set_elite's stored order (gaussian_mlp.py:363-379 index into it)
    layers = sm._layers()
    assert len(layers) == spec.num_layers + 1  # hidden layers + mean_and_logvar
    for li, layer in enumerate(layers):
        assert tuple(layer.weight.shape) == arrays["weights"][li].shape  # [E, K, N]
        assert tuple(layer.bias.shape) == arrays["biases"][li].shape    # [E, 1, N]
        np.testing.assert_array_equal(layer.weight.detach().numpy(), arrays["weights"][li])


@needs_ref
def test_signature_follows_training_side_mutations():
    spec, arrays, env = _real_model("halfcheetah_small")
    wrapper = env.dynamics_model
    sm = staging.StagedModel(wrapper, env.reward_fn, env.termination_fn, stage=False)
    s0 = sm._signature()
    assert sm._signature() == s0
    # ModelTrainer.train steps the optimiser in place (model_trainer.py:153) -> version counters move
    with torch.no_grad():
        wrapper.model.hidden_layers[1][0].weight.add_(1e-3)
    s1 = sm._signature()
    assert s1 != s0
    # set_elite replaces the elite list (model_trainer.py:288-296 -> gaussian_mlp.py:357-361)
    wrapper.set_elite([6, 5, 3, 2, 0][: spec.num_models])
    s2 = sm._signature()
    assert s2 != s1 and sm.members() == [6, 5, 3, 2, 0][: spec.num_models]
    # Normalizer.update_stats REPLACES mean / std tensors (util/math.py:114-127), via the wrapper's update_normalizer
    from mbrl.types import TransitionBatch

    rng = np.random.default_rng(0)
    n = 64
    batch = TransitionBatch(rng.standard_normal((n, spec.obs_dim)).astype(np.float32),
                            rng.standard_normal((n, spec.act_dim)).astype(np.float32),
                            rng.standard_normal((n, spec.obs_dim)).astype(np.float32),
                            np.zeros(n, np.float32), np.zeros(n, bool), np.zeros(n, bool))
    wrapper.update_normalizer(batch)
    s3 = sm._signature()
    assert s3 != s2
    # update_stats takes the dtype of the DATA (util/math.py:124-126): fp32 replay-buffer rows turn the "double precision"
    # normaliser's statistics into fp32 tensors, and normalize() then runs in fp32 -- staging follows the live tensors
    assert wrapper.input_normalizer.mean.dtype == torch.float32 and sm._describe().norm_mode == 1
    wrapper.input_normalizer.update_stats(torch.from_numpy(rng.standard_normal((n, spec.in_size))))  # fp64 rows
    assert sm._signature() != s3 and sm._describe().norm_mode == 2


def test_reference_callables_resolve_to_device_functions():
    rr, rt = RECORDED["reward_fns"], RECORDED["termination_fns"]
    for name in ("cartpole", "cartpole_pets", "inverted_pendulum", "halfcheetah", "pusher"):
        assert functions.resolve_reward(ref_surface.rebuild(rr[name])) == _lib.REWARD[name]
    for name in ("hopper", "cartpole", "inverted_pendulum", "no_termination", "walker2d", "ant", "humanoid"):
        assert functions.resolve_term(ref_surface.rebuild(rt[name])) == _lib.TERM[name]
    assert functions.resolve_reward(None) == _lib.REWARD["learned"]
    assert functions.resolve_reward(lambda a, o: o[:, :1]) == _lib.REWARD["external"]


@pytest.mark.parametrize("name", ["cem", "icem", "mppi"])
def test_shipped_optimizer_yaml_instantiates_into_b200_class(name, monkeypatch):
    """conf/action_optimizer/*.yaml carry `_target_: mbrl.planning.<X>Optimizer`, ${...} interpolations resolved here by
    hand (hydra does it in the reference, trajectory_opt.py:516-531 passes lower/upper bound itself)."""
    from mbrl_lib_b200 import planning

    cfg = RECORDED["optimizer_yaml"][name]
    assert cfg["_target_"].startswith("mbrl.planning.")
    resolved = {}
    for k, v in cfg.items():
        if isinstance(v, str) and v.startswith("${"):
            key = v.strip("${}").split(".")[-1]
            v = {"cem_num_iters": 5, "cem_elite_ratio": 0.1, "cem_population_size": 350, "cem_alpha": 0.1,
                 "cem_clipped_normal": False, "cem_population_decay_factor": 1.3, "cem_colored_noise_exponent": 2.0,
                 "cem_keep_elite_frac": 0.3, "mppi_num_iters": 5, "mppi_population_size": 350, "mppi_gamma": 0.9,
                 "mppi_sigma": 1.0, "mppi_beta": 0.9, "device": "cpu"}.get(key, v)
        if v == "???":
            continue
        resolved[k] = v
    H, A = 4, 2
    lower, upper = [[-1.0] * A] * H, [[1.0] * A] * H
    captured = {}

    # the classes need the library + a device at construction; record what _instantiate resolved instead
    for cls_name, cls in list(planning._KNOWN_TARGETS.items()):
        def fake(*a, _n=cls_name, **kw):
            captured["cls"], captured["kw"] = _n, kw
            return object()
        monkeypatch.setitem(planning._KNOWN_TARGETS, cls_name, fake)
    planning._instantiate(resolved, lower_bound=lower, upper_bound=upper)
    expect = {"cem": "CEMOptimizer", "icem": "ICEMOptimizer", "mppi": "MPPIOptimizer"}[name]
    assert captured["cls"] == expect
    # every key the YAML passes is a constructor argument of OUR class (same names as the reference's)
    import inspect

    real_cls = {"CEMOptimizer": planning.CEMOptimizer, "ICEMOptimizer": planning.ICEMOptimizer,
                "MPPIOptimizer": planning.MPPIOptimizer}[expect]
    ours = set(inspect.signature(real_cls.__init__).parameters) - {"self"}
    theirs = set(RECORDED["optimizer_ctor_args"][expect])
    assert set(captured["kw"]) <= ours, set(captured["kw"]) - ours
    assert theirs <= ours, f"reference ctor args missing from ours: {theirs - ours}"


@needs_ref
def test_classes_plug_into_reference_bases():
    """With mbrl importable when the package is first imported (a user's environment), Agent / Optimizer derive from
    mbrl.planning's own bases, so isinstance checks in user code keep working.  Own interpreter: import order matters."""
    import subprocess

    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "oracle", "ref_shims"), REF_SRC, ROOT])
    code = ("import mbrl.planning as rp, mbrl.planning.trajectory_opt as rt\n"
            "from mbrl_lib_b200 import planning as p\n"
            "assert issubclass(p.TrajectoryOptimizerAgent, rp.Agent)\n"
            "for c in (p.CEMOptimizer, p.ICEMOptimizer, p.MPPIOptimizer): assert issubclass(c, rt.Optimizer), c\n"
            "print('ok')")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


# ------------------------------------------------------------------------------------------------------------------
# GPU: our ModelEnv around the REAL reference model object vs the reference's ModelEnv on that same object
# ------------------------------------------------------------------------------------------------------------------
class _Feed:
    """torch.randperm / torch.normal return injected draws in call order (device tensors)."""

    def __init__(self, perms, normals):
        self.perms, self.normals = list(perms), list(normals)

    def __enter__(self):
        self._rp, self._nm = torch.randperm, torch.normal

        def randperm(n, **kw):
            p = self.perms.pop(0)
            assert p.numel() == n
            return p

        def normal(mean, std, *a, **kw):
            z = self.normals.pop(0)
            return mean + std * z

        torch.randperm, torch.normal = randperm, normal
        return self

    def __exit__(self, *a):
        torch.randperm, torch.normal = self._rp, self._nm


class _Box:
    def __init__(self, lo, hi, n):
        self.low, self.high, self.shape = np.full(n, lo, np.float32), np.full(n, hi, np.float32), (n,)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["halfcheetah_small", "cartpole", "hopper_tsinf", "pets_halfcheetah_small", "ant_learned_fn"])
@pytest.mark.parametrize("precision,tol", [("f32", 2e-4), ("bf16_tc", 2e-2)])
def test_our_model_env_on_real_reference_model_matches_reference_model_env(golden_dir, name, precision, tol):
    import mbrl_lib_b200 as bp

    dev = "cuda:0"
    spec, arrays, wrapper = _recorded_model(name, dev)
    inp = syn.make_rollout_inputs(spec)
    # the reference's ModelEnv.evaluate_action_sequences on its own object with these draws (oracle/gen_golden.py)
    gold = np.load(os.path.join(golden_dir, f"rollout_{name}.npz"))
    assert str(gold["model_sum"]) == syn.checksum(arrays) and str(gold["input_sum"]) == syn.checksum(inp)
    want = gold["returns"].astype(np.float32)
    acts = torch.from_numpy(inp["actions"]).to(dev)
    perms = torch.from_numpy(inp["perms"]).to(dev)
    eps = torch.from_numpy(inp["eps"]).to(dev)

    class _Env:
        observation_space = _Box(-np.inf, np.inf, spec.obs_dim)
        action_space = _Box(spec.action_lb, spec.action_ub, spec.act_dim)

    # ours, wrapping the reference's model object and its own reward / termination callables
    reward_fn, term_fn = _recorded_callables(spec)
    env = bp.ModelEnv(_Env(), wrapper, term_fn, reward_fn, generator=torch.Generator(device=dev), precision=precision,
                      ts1="perms")
    if precision == "bf16_tc" and not env.staged.supports_tc():
        pytest.skip("dims outside the tensor-core plan")
    got = env.evaluate_action_sequences(acts, inp["obs0"], spec.particles, _perms=perms, _eps=eps).cpu().numpy()
    scale = max(1.0, float(np.abs(want).max()))
    if spec.term_fn != "no_termination" or spec.reward_fn in ("cartpole",):
        frac = float((np.abs(got - want) > tol * scale).mean())
        assert frac <= 0.02, f"{frac:.3f} of sequences differ"
    else:
        np.testing.assert_allclose(got, want, atol=tol * scale, rtol=0)


@needs_ref
@pytest.mark.gpu
def test_training_pushes_weights_to_the_planner():
    """SURVEY.md 8f #3: after ModelEnv.hand_off_from(trainer), the reference's own ModelTrainer.train (Adam steps in place,
    best weights loaded back, set_elite; model_trainer.py:70-214, 288-296) leaves the packed device copy fresh WITHOUT any
    polling by act() / step(), and the planner evaluates exactly what the reference evaluates on the trained weights."""
    import mbrl_lib_b200 as bp
    from mbrl.types import TransitionBatch
    from mbrl.util.replay_buffer import BootstrapIterator, TransitionIterator

    dev = "cuda:0"
    spec, arrays, ref_env = _real_model("halfcheetah_small", dev)
    wrapper = ref_env.dynamics_model
    env = bp.ModelEnv(ref_env, wrapper, ref_env.termination_fn, ref_env.reward_fn, generator=torch.Generator(device=dev),
                      precision="f32", ts1="perms")
    trainer = mbrl.models.ModelTrainer(wrapper, optim_lr=1e-3, weight_decay=5e-5)
    env.hand_off_from(trainer)
    assert env._auto_refresh is False and env.staged._sig == env.staged._signature()

    rng = np.random.default_rng(3)
    n = 256
    obs = rng.standard_normal((n, spec.obs_dim)).astype(np.float32)
    act = rng.uniform(-1, 1, (n, spec.act_dim)).astype(np.float32)
    nxt = (obs + 0.1 * rng.standard_normal((n, spec.obs_dim))).astype(np.float32)
    data = TransitionBatch(obs, act, nxt, rng.standard_normal(n).astype(np.float32), np.zeros(n, bool), np.zeros(n, bool))
    wrapper.update_normalizer(data)  # wrapped: pushes
    assert env.staged._sig == env.staged._signature()
    sig0 = env.staged._sig
    train_it = BootstrapIterator(data, 64, spec.ensemble_size, shuffle_each_epoch=True, rng=rng)
    val_it = TransitionIterator(data, 64)
    trainer.train(train_it, dataset_val=val_it, num_epochs=2, silent=True)
    # the weights moved (Adam, in place), the elite list was re-ranked by validation score, and the copy followed -- pushed
    assert env.staged._sig != sig0
    assert env.staged._sig == env.staged._signature(), "training did not push its weights"
    assert env.staged.members() == list(wrapper.model.elite_models)

    inp = syn.make_rollout_inputs(spec)
    acts = torch.from_numpy(inp["actions"]).to(dev)
    perms = torch.from_numpy(inp["perms"]).to(dev)
    eps = torch.from_numpy(inp["eps"]).to(dev)
    with _Feed([perms[t] for t in range(perms.shape[0])], [eps[t] for t in range(spec.horizon)]):
        want = ref_env.evaluate_action_sequences(acts, inp["obs0"], spec.particles).float().cpu().numpy()
    calls = {"n": 0}
    real = env.staged.ensure_fresh

    def counting():
        calls["n"] += 1
        return real()

    env.staged.ensure_fresh = counting
    got = env.evaluate_action_sequences(acts, inp["obs0"], spec.particles, _perms=perms, _eps=eps).cpu().numpy()
    assert calls["n"] == 0, "the hot path still polls the parameters"
    np.testing.assert_allclose(got, want, atol=2e-4 * max(1.0, float(np.abs(want).max())), rtol=0)
