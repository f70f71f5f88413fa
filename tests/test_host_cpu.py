"""CPU-only checks of the host side: the C-ABI library loads and exports every symbol include/b200pets.h
declares, configuration plumbing mirrors the reference, and nothing silently falls back to the CPU."""
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from mbrl_lib_b200 import _lib

    header = open(os.path.join(ROOT, "include", "b200pets.h")).read()
    declared = set(re.findall(r"\b(b200pets_[a-z0-9_]+)\s*\(", header))
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in b200pets.h but not exported by libb200pets.so"
    assert declared == set(_lib.exported_symbols()), declared ^ set(_lib.exported_symbols())
    assert lib.b200pets_version() == 2


def test_no_cpu_fallback_for_models_on_cpu():
    import mbrl_lib_b200 as bp
    from mbrl_lib_b200 import functions, synthetic as syn

    spec = syn.CASES["halfcheetah_small"]
    model = bp.model_from_arrays(spec, syn.make_model_arrays(spec), "cpu")

    class _E:
        observation_space = None
        action_space = None

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        bp.ModelEnv(_E(), model, functions.no_termination, functions.reward_halfcheetah)


def test_callable_resolution():
    from mbrl_lib_b200 import _lib, functions

    assert functions.resolve_reward(None) == _lib.REWARD["learned"]
    assert functions.resolve_reward(functions.reward_halfcheetah) == _lib.REWARD["halfcheetah"]
    assert functions.resolve_term(functions.term_humanoid) == _lib.TERM["humanoid"]
    assert functions.resolve_reward(lambda a, o: o[:, :1]) == _lib.REWARD["external"]

    def halfcheetah(act, next_obs):  # stands in for mbrl.env.reward_fns.halfcheetah
        return next_obs[:, :1]

    halfcheetah.__module__ = "mbrl.env.reward_fns"
    assert functions.resolve_reward(halfcheetah) == _lib.REWARD["halfcheetah"]

    class HalfCheetahEnv:
        @staticmethod
        def preprocess_fn(s):
            return s

    assert functions.resolve_obs_process(HalfCheetahEnv.preprocess_fn) == _lib.PROC["halfcheetah"]
    with pytest.raises(NotImplementedError):
        functions.resolve_obs_process(lambda s: s)


def test_named_functions_match_oracle():
    from mbrl_lib_b200 import functions
    from oracle import pets_oracle as po

    g = torch.Generator().manual_seed(0)
    obs = torch.randn(64, 20, generator=g)
    obs[:, 0] = obs[:, 0].abs() + 0.5
    act = torch.randn(64, 7, generator=g)
    for name, fn in functions.REWARD_FNS.items():
        torch.testing.assert_close(fn(act, obs), po.REWARD_FNS[name](act, obs), rtol=1e-5, atol=1e-6)
    for name, fn in functions.TERM_FNS.items():
        assert torch.equal(fn(act, obs), po.TERM_FNS[name](act, obs))
    for name in ("halfcheetah", "cartpole"):
        torch.testing.assert_close(functions.OBS_PROCESS_FNS[name](obs), po.OBS_PROCESS[name](obs))


def test_icem_schedule_matches_reference_rule():
    import mbrl_lib_b200 as bp
    from oracle import pets_oracle as po

    lb, ub = [[-1.0] * 3] * 5, [[1.0] * 3] * 5
    for pop, decay, module in [(1000, 1.3, 7), (48, 1.3, 3), (500, 1.25, None)]:
        opt = bp.ICEMOptimizer(5, 0.1, pop, decay, 2.0, lb, ub, 0.3, 0.1, "cpu", population_size_module=module)
        assert opt.population_sizes() == po.icem_population_sizes(5, pop, decay, opt.elite_num, module)
    opt = bp.ICEMOptimizer(5, 0.1, 1000, 1.3, 2.0, lb, ub, 0.3, 0.1, "cpu", population_size_module=7)
    assert opt.elite_num == 100 and opt.keep_elite_size == 35  # SURVEY.md section 8 a4


def test_target_strings_select_b200_classes():
    from mbrl_lib_b200 import planning

    cfg = {"_target_": "mbrl.planning.CEMOptimizer", "num_iterations": 2, "elite_ratio": 0.1, "population_size": 10,
           "alpha": 0.1, "device": "cpu", "return_mean_elites": True}
    opt = planning._instantiate(cfg, lower_bound=[[-1.0]], upper_bound=[[1.0]])
    assert isinstance(opt, planning.CEMOptimizer) and opt.elite_num == 1
    to = planning.TrajectoryOptimizer(cfg, np.array([-1.0, -2.0]), np.array([1.0, 2.0]), planning_horizon=4)
    assert to.initial_solution.shape == (4, 2) and float(to.initial_solution.abs().max()) == 0.0
    assert to.optimizer.lower_bound.shape == (4, 2)


def test_staging_signature_tracks_training_side_changes():
    """weights mutate in place, normaliser tensors are replaced, elites change (SURVEY.md 3.4)."""
    import mbrl_lib_b200 as bp
    from mbrl_lib_b200 import synthetic as syn
    from mbrl_lib_b200.staging import StagedModel

    spec = syn.CASES["halfcheetah_small"]
    model = bp.model_from_arrays(spec, syn.make_model_arrays(spec), "cpu")
    st = StagedModel.__new__(StagedModel)
    st.src, st.mlp = model, model.model
    s0 = st._signature()
    with torch.no_grad():
        model.model.hidden_layers[1][0].weight.mul_(1.0)
    s1 = st._signature()
    model.input_normalizer.mean = model.input_normalizer.mean.clone()
    s2 = st._signature()
    model.set_elite([1, 2, 3, 4, 5])
    s3 = st._signature()
    assert len({s0, s1, s2, s3}) == 4


def test_staging_reads_the_real_reference_objects():
    """Drop-in check against mbrl-lib's own classes, as recorded from the imported reference (oracle/gen_golden.py,
    oracle/ref_surface.py): the staging code must find every attribute it needs on OneDTransitionRewardModel(GaussianMLP)
    -- GaussianMLP(23, 17, SiLU, 4 x 200, ensemble 7), fp64 normaliser, set_elite([0, 2, 3, 5, 6]) -- and resolve
    mbrl's own reward / termination fns."""
    import json

    from mbrl_lib_b200 import _lib, functions
    from mbrl_lib_b200.staging import StagedModel
    from oracle import ref_surface

    with open(os.path.join(ROOT, "tests", "golden", "reference_objects.json")) as f:
        rec = json.load(f)
    R = {k: ref_surface.rebuild(v) for k, v in rec["reward_fns"].items()}
    T = {k: ref_surface.rebuild(v) for k, v in rec["termination_fns"].items()}
    wrapper = ref_surface.rebuild(rec["models"]["silu_fp64_normalizer"])
    st = StagedModel.__new__(StagedModel)
    st.src, st.mlp = wrapper, wrapper.model
    st.reward_id = functions.resolve_reward(R["halfcheetah"])
    st.term_id = functions.resolve_term(T["no_termination"])
    d = st._describe()
    assert (d.ensemble_size, d.num_members, d.obs_dim, d.act_dim, d.in_size, d.out_size, d.hid_size, d.num_hidden) == \
        (7, 5, 17, 6, 23, 17, 200, 4)
    assert d.activation == _lib.ACT["silu"] and d.norm_mode == 2 and d.target_is_delta == 1 and d.learned_rewards == 0
    assert d.reward_fn == _lib.REWARD["halfcheetah"] and d.term_fn == _lib.TERM["no_termination"]
    assert st.members() == [0, 2, 3, 5, 6]
    assert [tuple(l.weight.shape) for l in st._layers()] == [(7, 23, 200)] + [(7, 200, 200)] * 3 + [(7, 200, 34)]
    for name in ("cartpole", "cartpole_pets", "inverted_pendulum", "pusher"):
        assert functions.resolve_reward(R[name]) == _lib.REWARD[name]
    for name in ("hopper", "cartpole", "inverted_pendulum", "walker2d", "ant", "humanoid"):
        assert functions.resolve_term(T[name]) == _lib.TERM[name]


def test_rollout_model_env_protocol():
    """Same protocol the reference checks in tests/core/test_common_utils.py:195-227, with stand-in env / agent."""
    from mbrl_lib_b200.planning import rollout_model_env

    class _CountingEnv:
        def reset(self, obs0, return_as_np=None):
            self.obs, self.kw = obs0, return_as_np
            return {}

        def step(self, action, model_state, sample=None):
            assert sample is False
            self.obs = self.obs + action[:, :1]
            n = self.obs.shape[0]
            return self.obs, np.ones(n), np.zeros(n), {}

    class _FixedAgent:
        def __init__(self, n):
            self.seq = np.ones((n, 1))

        def plan(self, obs):
            assert obs.ndim == 2  # the reference hands the agent a [1, D] observation
            return self.seq

    env, agent, D, L, S = _CountingEnv(), _FixedAgent(12), 7, 12, 3
    obs, rew, plan = rollout_model_env(env, np.zeros(D), 0 * agent.seq, agent, num_samples=S)  # agent wins over plan
    assert env.kw is True and obs.shape == (L + 1, S, D) and rew.shape == (L, S) and plan.shape == (L, 1)
    assert [o.min() for o in obs] == list(range(L + 1))
    obs, _, _ = rollout_model_env(env, np.zeros(D), 3 * agent.seq, None, num_samples=S)
    assert [o.max() for o in obs] == [3 * i for i in range(L + 1)]


def test_hand_off_wrappers_push_every_registered_env():
    """ModelEnv.hand_off_from: wrapping is idempotent per object and serves several environments of one model (CPU: the
    environments are bare objects with a counting stand-in for the staged copy; the GPU test runs the reference's trainer)."""
    from mbrl_lib_b200.model_env import ModelEnv

    class _Staged:
        def __init__(self):
            self.n = 0

        def ensure_fresh(self):
            self.n += 1

    class _Model:
        def __init__(self):
            self.calls = []

        def update_normalizer(self, batch):
            self.calls.append("norm")

        def set_elite(self, idx):
            self.calls.append("elite")

    class _Trainer:
        def train(self, *a, **kw):
            return "losses"

    def bare_env(model):
        e = ModelEnv.__new__(ModelEnv)
        e.dynamics_model, e.staged, e._auto_refresh = model, _Staged(), True
        return e

    model, trainer = _Model(), _Trainer()
    e1, e2 = bare_env(model), bare_env(model)
    assert e1.hand_off_from(trainer) is trainer and e1._auto_refresh is False and e1.staged.n == 1
    e1.hand_off_from(trainer)  # again: no second layer of wrappers
    e2.hand_off_from(trainer)
    n1, n2 = e1.staged.n, e2.staged.n
    assert trainer.train("data") == "losses"
    assert (e1.staged.n, e2.staged.n) == (n1 + 1, n2 + 1), "one push per environment and call"
    model.update_normalizer(None)
    model.set_elite([0])
    assert model.calls == ["norm", "elite"] and (e1.staged.n, e2.staged.n) == (n1 + 3, n2 + 3)
    e1._fresh()  # the hot path no longer polls
    assert e1.staged.n == n1 + 3
