"""The oracle (oracle/pets_oracle.py) against golden vectors produced by the imported reference
(oracle/gen_golden.py).  CPU only.  These pin the checker before it is trusted to judge the CUDA path."""
import os

import numpy as np
import pytest
import torch

from mbrl_lib_b200 import synthetic as syn
from oracle import pets_oracle as po

ROLLOUT_CASES = ["cartpole", "halfcheetah", "halfcheetah_small", "pets_halfcheetah_small", "humanoid_trunc",
                 "relu_expectation", "silu_expectation", "hopper_tsinf", "cartpole_pets", "pusher_det", "walker_ant", "humanoid_v4", "tc_hid64", "tc_wide", "tc_shallow", "ant_learned_fn"]


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name), allow_pickle=False)


@pytest.mark.parametrize("name", ROLLOUT_CASES)
def test_rollout_matches_reference(golden_dir, name):
    spec = syn.CASES[name]
    arrays = syn.make_model_arrays(spec)
    inp = syn.make_rollout_inputs(spec)
    g = _load(golden_dir, f"rollout_{name}.npz")
    assert str(g["model_sum"]) == syn.checksum(arrays), "regenerated weights differ from the golden run's"
    assert str(g["input_sum"]) == syn.checksum(inp), "regenerated inputs differ from the golden run's"
    m = po.OracleModel(spec, arrays)
    ret = m.evaluate_action_sequences(torch.from_numpy(inp["actions"]), inp["obs0"], spec.particles,
                                      torch.from_numpy(inp["perms"]), torch.from_numpy(inp["eps"]))
    # same ATen ops as the reference => bit-exact here; 1e-6 leaves room for a different MKL thread split
    np.testing.assert_allclose(ret.numpy(), g["returns"], rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("name", ROLLOUT_CASES)
def test_float64_oracle_matches_reference(golden_dir, name):
    """The double-precision oracle (the yardstick of tests/test_gpu_shapes.py) differs from the reference's fp32
    arithmetic by rounding only: 1e-5 of the return scale on every golden rollout."""
    spec = syn.CASES[name]
    arrays = syn.make_model_arrays(spec)
    inp = syn.make_rollout_inputs(spec)
    g = _load(golden_dir, f"rollout_{name}.npz")
    m = po.OracleModel(spec, arrays, dtype=torch.float64)
    ret = m.evaluate_action_sequences(torch.from_numpy(inp["actions"]), inp["obs0"], spec.particles,
                                      torch.from_numpy(inp["perms"]), torch.from_numpy(inp["eps"]))
    assert ret.dtype == torch.float64
    scale = max(1.0, float(np.abs(g["returns"]).max()))
    err = float(np.abs(ret.numpy() - g["returns"]).max())
    assert err <= 1e-5 * scale, f"max |diff| {err:.3e} > 1e-5 * {scale:.3g}"


@pytest.mark.parametrize("name,batch", [("mbpo_halfcheetah_small", 1000), ("cartpole", 500)])
def test_float64_oracle_step_matches_reference(golden_dir, name, batch):
    spec = syn.CASES[name]
    arrays = syn.make_model_arrays(spec)
    inp = syn.make_step_inputs(spec, batch)
    g = _load(golden_dir, f"step_{name}.npz")
    m = po.OracleModel(spec, arrays, dtype=torch.float64)
    nobs, rew, done = m.step(torch.from_numpy(inp["obs"]), torch.from_numpy(inp["act"]),
                             torch.from_numpy(inp["perm"]), torch.from_numpy(inp["eps"]))
    scale = max(1.0, float(np.abs(g["next_obs"]).max()))
    assert np.abs(nobs.numpy() - g["next_obs"]).max() <= 1e-5 * scale
    assert np.abs(rew.numpy() - g["reward"]).max() <= 1e-5 * scale
    assert (done.numpy() == g["done"]).all()


def test_float64_bf16_emulation_keeps_double_accumulation():
    """emulate_bf16 in fp64 mode rounds the operands (activations, weights, the two bias parts) to bf16 and nothing
    else: products and sums stay in double.  Restated layer by layer with numpy float64."""
    x = torch.tensor([1.0 + 2.0 ** -7, 1.0 + 2.0 ** -9], dtype=torch.float64)
    assert po._bf16_round(x).dtype == torch.float64
    assert po._bf16_round(x).tolist() == [1.0 + 2.0 ** -7, 1.0]  # 8 significant bits, round to nearest even
    spec = syn.CASES["tc_hid64"]
    arrays = syn.make_model_arrays(spec)
    m = po.OracleModel(spec, arrays, dtype=torch.float64)
    m.emulate_bf16 = True
    xs = torch.randn(len(m.members), 16, spec.in_size, generator=torch.Generator().manual_seed(0), dtype=torch.float64)
    mean, lv = m.mlp(xs)
    assert mean.dtype == torch.float64 and lv.dtype == torch.float64

    def bf(a):
        return torch.from_numpy(np.asarray(a, np.float64)).to(torch.bfloat16).double().numpy()

    h = xs.numpy()
    for li, (w, b) in enumerate(zip(arrays["weights"], arrays["biases"])):
        w, b = w[m.members].astype(np.float64), b[m.members].astype(np.float64)
        h = np.matmul(bf(h), bf(w)) + (bf(b) + bf(b - bf(b)))
        if li < len(arrays["weights"]) - 1:
            h = h / (1.0 + np.exp(-h))  # SiLU
    np.testing.assert_allclose(mean.numpy(), h[..., :spec.out_size], rtol=1e-12, atol=1e-12)
    m32 = po.OracleModel(spec, arrays)
    m32.emulate_bf16 = True
    mean32, _ = m32.mlp(xs.float())
    assert not np.array_equal(mean32.double().numpy(), mean.numpy())  # fp32 accumulation rounds differently


def test_full_elite_list_keeps_member_order():
    """GaussianMLP.set_elite (gaussian_mlp.py:377-379) ignores an elite list as long as the ensemble: a reordered full
    list runs the members in index order, exactly like no list."""
    import dataclasses

    base = dataclasses.replace(syn.CASES["tc_hid64"], elites=None)
    arrays = syn.make_model_arrays(base)
    inp = syn.make_rollout_inputs(base)
    args = (torch.from_numpy(inp["actions"]), inp["obs0"], base.particles, torch.from_numpy(inp["perms"]),
            torch.from_numpy(inp["eps"]))
    ref = po.OracleModel(base, arrays).evaluate_action_sequences(*args)
    full = po.OracleModel(dataclasses.replace(base, elites=(2, 0, 1)), arrays)
    assert full.members == [0, 1, 2]
    assert torch.equal(full.evaluate_action_sequences(*args), ref)
    assert po.OracleModel(dataclasses.replace(base, elites=(2, 0)), arrays).members == [2, 0]  # a true subset keeps its order


@pytest.mark.parametrize("name", ["halfcheetah_small", "hopper_tsinf", "ant_learned_fn", "tc_hid64"])
def test_assigned_members_path_equals_permutation_path(name):
    """``forward_assigned`` (row -> member map given directly; what the GPU tile-shuffle tests feed the oracle) equals the
    golden-pinned permutation path for the map a permutation induces (gaussian_mlp.py:202-212)."""
    spec = syn.CASES[name]
    arrays = syn.make_model_arrays(spec)
    inp = syn.make_rollout_inputs(spec)
    m = po.OracleModel(spec, arrays)
    args = (torch.from_numpy(inp["actions"]), inp["obs0"], spec.particles)
    ref = m.evaluate_action_sequences(*args, torch.from_numpy(inp["perms"]), torch.from_numpy(inp["eps"])).numpy()
    B, M = spec.batch, spec.num_models
    assign = np.empty(inp["perms"].shape, np.int64)
    for t in range(assign.shape[0]):
        assign[t, inp["perms"][t]] = np.arange(B) // (B // M)
    got = m.evaluate_action_sequences(*args, None, torch.from_numpy(inp["eps"]), assign=torch.from_numpy(assign)).numpy()
    np.testing.assert_allclose(got, ref, rtol=1e-5, atol=1e-5)  # only the GEMM batch split differs


@pytest.mark.parametrize("name,batch", [("mbpo_halfcheetah_small", 1000), ("cartpole", 500)])
def test_step_matches_reference(golden_dir, name, batch):
    spec = syn.CASES[name]
    arrays = syn.make_model_arrays(spec)
    inp = syn.make_step_inputs(spec, batch)
    g = _load(golden_dir, f"step_{name}.npz")
    assert str(g["input_sum"]) == syn.checksum(inp)
    m = po.OracleModel(spec, arrays)
    nobs, rew, done = m.step(torch.from_numpy(inp["obs"]), torch.from_numpy(inp["act"]),
                             torch.from_numpy(inp["perm"]), torch.from_numpy(inp["eps"]))
    np.testing.assert_allclose(nobs.numpy(), g["next_obs"], rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(rew.numpy(), g["reward"], rtol=1e-6, atol=1e-6)
    assert (done.numpy() == g["done"]).all()


def _quad(target):
    return lambda pop, i: -((pop - target) ** 2).sum(dim=(1, 2)) + 0.3 * torch.sin(3.0 * pop).sum(dim=(1, 2))


@pytest.mark.parametrize("tag,clipped,ret_mean", [("trunc_best", False, False), ("trunc_mean", False, True),
                                                  ("clipped_best", True, False)])
def test_cem_matches_reference(golden_dir, tag, clipped, ret_mean):
    g = _load(golden_dir, f"cem_{tag}.npz")
    t = lambda k: torch.from_numpy(g[k])  # noqa: E731
    trace = []
    sol = po.cem_optimize(_quad(t("target")), t("x0"), t("lb"), t("ub"), int(g["iters"]), float(g["elite_ratio"]),
                          int(g["N"]), float(g["alpha"]), t("z"), return_mean_elites=ret_mean,
                          clipped_normal=clipped, trace=trace)
    for i, tr in enumerate(trace):
        np.testing.assert_allclose(tr["pop"].numpy(), g["pops"][i], rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(tr["values"].numpy(), g["values"][i], rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(sol.numpy(), g["solution"], rtol=1e-6, atol=1e-7)


def test_icem_matches_reference(golden_dir):
    g = _load(golden_dir, "icem.npz")
    t = lambda k: torch.from_numpy(g[k])  # noqa: E731
    iters = int(g["iters"])
    elite = None
    for call in range(2):
        noise = []
        for i in range(iters):
            d = {"sr": t(f"c{call}_sr{i}"), "si": t(f"c{call}_si{i}")}
            if f"c{call}_perm{i}" in g:
                d["keep_perm"] = t(f"c{call}_perm{i}")
            if i == 0 and f"c{call}_end_eps" in g:
                d["end_eps"] = t(f"c{call}_end_eps")
            noise.append(d)
        trace = []
        sol, elite = po.icem_optimize(_quad(t("target")), t("x0"), t("lb"), t("ub"), iters, float(g["elite_ratio"]),
                                      int(g["pop0"]), float(g["decay"]), float(g["beta"]), float(g["keep_frac"]),
                                      float(g["alpha"]), noise, prev_elite=elite, module=int(g["module"]), trace=trace)
        for i, tr in enumerate(trace):
            np.testing.assert_allclose(tr["pop"].numpy(), g[f"c{call}_pop{i}"], rtol=1e-5, atol=1e-6)
            np.testing.assert_allclose(tr["values"].numpy(), g[f"c{call}_val{i}"], rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(sol.numpy(), g[f"sol{call}"], rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(elite.numpy(), g[f"c{call}_elite"], rtol=1e-5, atol=1e-6)


def test_mppi_matches_reference(golden_dir):
    g = _load(golden_dir, "mppi.npz")
    t = lambda k: torch.from_numpy(g[k])  # noqa: E731
    H, A = g["lb"].shape
    mean = torch.zeros(H, A)
    for call in range(2):
        trace = []
        mean = po.mppi_optimize(_quad(t("target")), mean, t("lb"), t("ub"), int(g["iters"]), int(g["N"]), float(g["gamma"]),
                                float(g["beta"]), t(f"z{call}"), trace=trace)
        for k, tr in enumerate(trace):
            np.testing.assert_allclose(tr["pop"].numpy(), g[f"pops{call}"][k], rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(mean.numpy(), g[f"sol{call}"], rtol=1e-6, atol=1e-7)


def test_cem_over_model_matches_reference(golden_dir):
    g = _load(golden_dir, "cem_model.npz")
    spec = syn.CASES["halfcheetah_small"]
    arrays = syn.make_model_arrays(spec)
    inp = syn.make_rollout_inputs(spec)
    iters = int(g["iters"])
    nz = syn.make_cem_noise(spec, iters)
    assert str(g["noise_sum"]) == syn.checksum(nz)
    m = po.OracleModel(spec, arrays)
    H, A = spec.horizon, spec.act_dim
    lb = torch.full((H, A), spec.action_lb)
    ub = torch.full((H, A), spec.action_ub)

    def obj(pop, i):
        return m.evaluate_action_sequences(pop, inp["obs0"], spec.particles, torch.from_numpy(nz["perms"][i]),
                                           torch.from_numpy(nz["eps"][i]))

    trace = []
    sol = po.cem_optimize(obj, torch.zeros(H, A), lb, ub, iters, 0.1, spec.population, 0.1,
                          torch.from_numpy(nz["z"]), return_mean_elites=True, trace=trace)
    for i, tr in enumerate(trace):
        np.testing.assert_allclose(tr["values"].numpy(), g["values"][i], rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(sol.numpy(), g["solution"], rtol=1e-6, atol=1e-7)


def test_reference_known_answer_dummy_model(golden_dir):
    """The reference's only known-answer test of evaluate_action_sequences (tests/core/test_models.py:365-385):
    next_obs = obs + act, reward = next_obs  =>  return = H(H+1)/2 * a.  The dummy model is expressed as a
    hand-built ReLU ensemble (synthetic.counter_world) so the whole oracle path runs: model input, member
    routing by permutation, delta targets, learned-reward column, accumulation and the particle mean."""
    spec, arrays = syn.counter_world()
    gold = _load(golden_dir, "kat_counter_world.npz")  # the imported reference on the same hand-built model
    assert str(gold["model_sum"]) == syn.checksum(arrays)
    m = po.OracleModel(spec, arrays)
    g = np.random.default_rng(0)
    N = 4
    for P in range(1, 10):
        for H in range(1, 10):
            for a in (1.0, 2.0):
                B = N * P
                actions = torch.full((N, H, 1), a)
                perms = torch.from_numpy(np.stack([g.permutation(B) for _ in range(H)]))
                for bf16 in (False, True):
                    m.emulate_bf16 = bf16
                    ret = m.evaluate_action_sequences(actions, np.zeros(1), P, perms, None)
                    assert torch.equal(ret, torch.full((N,), H * (H + 1) / 2 * a)), (P, H, a, bf16)
                    assert ret[0].item() == gold["returns"][P - 1, H - 1, int(a) - 1]


def test_bf16_emulation_tolerance_band():
    """How far bf16 operands (fp32 accumulate) move per-sequence returns at the headline config: this is the
    measured justification of the tolerance the tensor-core parity tests state."""
    spec = syn.CASES["halfcheetah_small"]
    arrays = syn.make_model_arrays(spec)
    inp = syn.make_rollout_inputs(spec)
    m = po.OracleModel(spec, arrays)
    args = (torch.from_numpy(inp["actions"]), inp["obs0"], spec.particles, torch.from_numpy(inp["perms"]),
            torch.from_numpy(inp["eps"]))
    r32 = m.evaluate_action_sequences(*args)
    m.emulate_bf16 = True
    r16 = m.evaluate_action_sequences(*args)
    err = (r16 - r32).abs().max().item()
    scale = r32.abs().max().item()
    assert err <= 2e-2 * max(scale, 1.0), (err, scale)
