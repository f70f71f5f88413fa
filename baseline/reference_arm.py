"""Reference arm of bench.py: the UNMODIFIED reference (facebookresearch/mbrl-lib) on the host CPUs.

The package is imported from ``oracle/_ref`` (the copy ``build()`` makes with ``oracle/ref_install.py``) or from
``baseline/_ref`` (a ``pip install --no-deps --target`` of mbrl-lib); both are git-ignored.  mbrl-lib imports hydra, omegaconf,
gymnasium and termcolor at module level; none of them is installed in this image and there is no index, so the
API shims under ``oracle/ref_shims`` (a dict-backed DictConfig, ``hydra.utils.instantiate``, ``gymnasium.spaces.Box``)
stand in for them.  They are configuration plumbing only: every tensor operation on the timed path
(``TrajectoryOptimizerAgent.act`` -> ``CEMOptimizer.optimize`` -> ``ModelEnv.evaluate_action_sequences`` ->
``OneDTransitionRewardModel`` -> ``GaussianMLP``) is the reference's own code.

Nothing in the product imports this module; bench.py's ``--impl reference`` and ``cpu_baseline`` legs do.
"""
from __future__ import annotations

import importlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ACT = {"relu": "torch.nn.ReLU", "silu": "torch.nn.SiLU", "leaky_relu": "torch.nn.LeakyReLU"}


def import_reference():
    """Returns (mbrl package, where it came from) or (None, reason)."""
    if "mbrl" in sys.modules and hasattr(sys.modules["mbrl"], "__b200_ref_source__"):
        return sys.modules["mbrl"], sys.modules["mbrl"].__b200_ref_source__
    shims = os.path.join(ROOT, "oracle", "ref_shims")
    for missing in ("hydra", "omegaconf", "gymnasium", "termcolor"):
        try:
            importlib.import_module(missing)
        except ImportError:
            if shims not in sys.path:
                sys.path.insert(0, shims)
    for cand in (os.path.join(ROOT, "oracle", "_ref"), os.path.join(ROOT, "baseline", "_ref")):
        if os.path.isdir(os.path.join(cand, "mbrl")):
            sys.path.insert(0, cand)
            try:
                mbrl = importlib.import_module("mbrl")
                importlib.import_module("mbrl.models")
                importlib.import_module("mbrl.planning")
                importlib.import_module("mbrl.env.reward_fns")
                importlib.import_module("mbrl.env.termination_fns")
                mbrl.__b200_ref_source__ = cand
                return mbrl, cand
            except Exception as e:  # pragma: no cover - depends on the box
                sys.path.remove(cand)
                for k in [k for k in sys.modules if k == "mbrl" or k.startswith("mbrl.")]:
                    del sys.modules[k]
                last = f"{cand}: {type(e).__name__}: {e}"
                continue
    return None, locals().get("last", "no oracle/_ref and no baseline/_ref")


def _proc_fn(name):
    if name is None:
        return None
    if name == "halfcheetah":  # mbrl/env/pets_halfcheetah.py:91-113 (the module itself needs mujoco)
        return lambda s: torch.cat([s[..., 1:2], torch.sin(s[..., 2:3]), torch.cos(s[..., 2:3]), s[..., 3:]], dim=-1)
    if name == "cartpole":  # mbrl/env/pets_cartpole.py:78-101
        return lambda s: torch.cat([torch.sin(s[..., 1:2]), torch.cos(s[..., 1:2]), s[..., :1], s[..., 2:]], dim=-1)
    raise ValueError(name)


class _Env:
    def __init__(self, spec):
        import gymnasium

        self.observation_space = gymnasium.spaces.Box(-np.inf, np.inf, (spec.obs_dim,))
        self.action_space = gymnasium.spaces.Box(spec.action_lb, spec.action_ub, (spec.act_dim,))


def build_model_env(mbrl, spec, arrays, seed: int = 0):
    """The reference's GaussianMLP + OneDTransitionRewardModel + ModelEnv carrying the synthetic weights of ``spec``."""
    import mbrl.env.reward_fns as ref_rew
    import mbrl.env.termination_fns as ref_term

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
        obs_process_fn=_proc_fn(spec.obs_process), no_delta_list=list(spec.no_delta_list), num_elites=spec.num_models)
    if spec.normalize is not None:
        wrapper.input_normalizer.mean = torch.from_numpy(arrays["norm_mean"])
        wrapper.input_normalizer.std = torch.from_numpy(arrays["norm_std"])
    if spec.elites is not None:
        wrapper.set_elite(list(spec.elites))
    reward_fn = getattr(ref_rew, spec.reward_fn) if spec.reward_fn else None
    term_fn = getattr(ref_term, spec.term_fn)
    return mbrl.models.ModelEnv(_Env(spec), wrapper, term_fn, reward_fn, generator=torch.Generator().manual_seed(seed))


def build_agent(mbrl, model_env, spec, iters: int, elite_ratio: float, alpha: float, population: int = 0):
    """``mbrl.planning.create_trajectory_optim_agent_for_model`` with the shipped cem.yaml's keys
    (mbrl/examples/conf/action_optimizer/cem.yaml, mbrl/planning/trajectory_opt.py:719-749)."""
    import omegaconf

    cfg = omegaconf.OmegaConf.create({
        "_target_": "mbrl.planning.TrajectoryOptimizerAgent", "planning_horizon": spec.horizon, "replan_freq": 1,
        "verbose": False,
        "action_lb": [float(spec.action_lb)] * spec.act_dim, "action_ub": [float(spec.action_ub)] * spec.act_dim,
        "optimizer_cfg": {"_target_": "mbrl.planning.CEMOptimizer", "num_iterations": iters, "elite_ratio": elite_ratio,
                          "population_size": population or spec.population, "alpha": alpha, "device": "cpu",
                          "lower_bound": "???", "upper_bound": "???", "return_mean_elites": True,
                          "clipped_normal": False}})
    return mbrl.planning.create_trajectory_optim_agent_for_model(model_env, cfg, num_particles=spec.particles)
