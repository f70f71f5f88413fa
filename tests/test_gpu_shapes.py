"""Shape sweep: both rollout kernels against the float64 oracle across the code paths the model shape selects.

The tensor-core kernel (csrc/rollout_tc.cu) picks its epilogue branches from the hidden width, the input width, the output
width, the depth and the activation; the fp32 kernel (csrc/rollout_f32.cu) picks its row tile from the shared-memory
footprint.  The cases below are generated ``synthetic.CaseSpec`` objects (not registered in ``synthetic.CASES``: the
goldens and their checksums do not depend on them), small enough that the float64 oracle runs in seconds.  Which branch
each case reaches is restated in Python (``tc_plan`` / ``f32_rows``, each predicate next to the kernel line it mirrors);
``tests/test_shape_coverage.py`` (CPU) checks that the table covers every branch, ``test_plan_restatement_matches_library``
(GPU) that the restatement agrees with the library's own plan.

Modes, on both kernels wherever the tensor-core plan accepts the shape:
  ts1      TS1, injected per-step permutations and model noise
  tsinf    TSinf (propagation "fixed_model"), one injected reset permutation
  shuffle  the in-kernel tile shuffle, checked with the exported member map (as tests/test_gpu_shuffle.py)
  expect   propagation "expectation" (a subset)
Bars (tests/test_gpu_parity.py): fp32 kernel |diff| <= 2e-4 * scale against the float64 oracle; tensor-core kernel
<= 5e-3 * scale against the float64 oracle with bf16-rounded operands; the discrete-reward case by the discrete bars.

The multi-tile cases size the grid to at least twice the SM count with a partial last tile, so every CTA of the persistent
tensor-core kernel carries barrier parities, weight-ring stage / phase, the activation-buffer counter and the tail
constants from one tile into the next.
"""
import ctypes as C
import dataclasses

import numpy as np
import pytest
import torch

from mbrl_lib_b200 import synthetic as syn

DEV = "cuda:0"
B200_SMS = 148
MAX_SMEM_OPTIN = 232448  # cudaDevAttrMaxSharedMemoryPerBlockOptin on sm_100


def _r16(x):
    return (x + 15) // 16 * 16


# ---- restatement of the plan choices ---------------------------------------------------------------------------------
def tc_plan(s, expectation=False, max_smem=MAX_SMEM_OPTIN):
    """tc_make_plan (rollout_tc.cu:1288-1345) and the kernel's branch predicates; None where the plan rejects the shape."""
    L, D, Dp, A, inn, hid, out = s.num_layers, s.obs_dim, s.proc_obs_dim, s.act_dim, s.in_size, s.hid_size, s.out_size
    nout = out if s.deterministic else 2 * out                                   # api.cu:212
    outp = _r16(out)                                                             # api.cu:216
    Kp = [_r16(k + 2) for k in [inn] + [hid] * L]                                # api.cu:224
    Np = [_r16(hid)] * L + [outp if s.deterministic else 2 * outp]               # api.cu:225
    if inn + 2 > 256 or hid + 2 > 256 or nout > 256 or D > 256:                  # rollout_tc.cu:1291
        return None
    if max(Kp) > 256 or max(Np) > 256:                                           # rollout_tc.cu:1295
        return None
    stage = (max(k * n * 2 for k, n in zip(Kp, Np)) + 127) & ~127                # rollout_tc.cu:1298-1301
    C_ = Np[0] // 16
    h0n = 16 * max(1, min(C_ - 1, (C_ * 8 + 6) // 13))                           # rollout_tc.cu:1308-1313
    if Np[0] - h0n < 16:                                                         # rollout_tc.cu:1315
        return None
    outq = (out + 3) & ~3
    al16 = lambda x: (x + 15) & ~15  # noqa: E731
    off = 128 * (max(D, outq) | 1) * 4 + 3 * 128 * (A | 1) * 4                   # rollout_tc.cu:1319-1324
    off = al16(off + 128 * ((Kp[0] - Dp) | 1) * 4)                               # rollout_tc.cu:1325-1327
    off = al16(off + 2 * Kp[0] * 4)
    off = al16(off + 4 * outq * 4)
    if expectation:
        off += 128 * ((2 * outq) | 1) * 4                                        # rollout_tc.cu:1334
    off = al16(off)
    off = (off + (2 * 8 + 4) * 8 + 16 + 127) & ~127                              # rollout_tc.cu:1336-1337
    S = (max_smem - off) // stage                                                # rollout_tc.cu:1339
    if S < 1:
        return None
    c_tail = Np[0] // 16 - 1
    return dict(
        Kp0=Kp[0], h0n=h0n, nstages=min(S, 8), smem=off + min(S, 8) * stage,
        fast_tail=L >= 1 and hid - 16 * c_tail == 8 and hid >= Kp[0],            # rollout_tc.cu:523
        final_early=Np[L] <= h0n,                                                # rollout_tc.cu:381
        fuse_in=L >= 4 and not expectation and s.obs_process is None and s.horizon >= 2,  # rollout_tc.cu:510, 761
        act_regs=A <= 8,                                                         # rollout_tc.cu:565 (injected actions)
    )


def f32_rows(s, max_smem=MAX_SMEM_OPTIN):
    """Row tile of the fp32 kernel: the largest of 64 / 32 / 16 whose footprint fits (rollout_f32.cu:308-332)."""
    nout = s.out_size if s.deterministic else 2 * s.out_size
    LD = ((max(s.in_size, s.hid_size, nout) + 3) & ~3) + 4                        # rollout_f32.cu:309-311
    for TR in (64, 32, 16):
        if TR * (2 * LD + s.obs_dim + s.act_dim + nout + 2) * 4 + TR * (2 * 8 + 4) <= max_smem:  # rollout_f32.cu:312-314
            return TR
    return None


def tc_tiles(s, mode):
    """Tiles of one tensor-core launch (rollout_tc.cu:1361-1369)."""
    B = s.population * s.particles
    if mode == "expect":
        return -(-B // 128)
    if mode == "shuffle":
        return s.particles * -(-s.population // 128)
    return s.num_models * -(-(B // s.num_models) // 128)


# ---- the case table ---------------------------------------------------------------------------------------------------
def _case(name, obs, act, hid, L, activation, *, ens=3, elites=None, pop=30, H=5, P=3, **kw):
    return syn.CaseSpec(f"sweep_{name}", obs_dim=obs, act_dim=act, hid_size=hid, num_layers=L, ensemble_size=ens,
                        elites=elites, activation=activation, population=pop, horizon=H, particles=P,
                        **{"normalize": None, "reward_fn": "halfcheetah", "term_fn": "no_termination", **kw})


# name -> (spec, modes).  Continuous rewards, no termination (the exact bars) unless stated.
SWEEP = {c.name[len("sweep_"):]: (c, m) for c, m in [
    (_case("h17_L1", 5, 2, 17, 1, "relu", pop=30, P=3, H=5), ("ts1", "tsinf", "shuffle", "expect")),  # smallest width
    (_case("h18_L2", 6, 3, 18, 2, "leaky_relu", ens=4, elites=(1, 3), pop=40, P=4, H=6, normalize="float32"),
     ("ts1", "tsinf", "shuffle")),
    (_case("h35_L3", 7, 2, 35, 3, "silu", pop=33, P=5, H=7, normalize="float64"), ("ts1", "tsinf", "shuffle", "expect")),
    (_case("h52_L4_relu", 8, 4, 52, 4, "relu", ens=5, elites=(0, 2, 4), pop=45, P=4, H=6, normalize="float64"),
     ("ts1", "tsinf", "shuffle")),
    (_case("h69_L5_leaky_a9", 11, 9, 69, 5, "leaky_relu", ens=4, pop=48, P=3, H=5, normalize="float32"),
     ("ts1", "tsinf", "shuffle", "expect")),
    (_case("h86_L6_det", 13, 3, 86, 6, "silu", pop=36, P=3, H=6, deterministic=True), ("ts1", "tsinf", "shuffle")),
    (_case("h103_L7_abs", 17, 6, 103, 7, "silu", ens=5, elites=(4, 1, 2, 0, 3), pop=50, P=5, H=7, normalize="float64",
           target_is_delta=False), ("ts1", "tsinf", "shuffle")),
    (_case("h40_slow_tail", 40, 6, 40, 2, "silu", pop=30, P=4, H=5, normalize="float64"), ("ts1", "tsinf", "shuffle")),
    (_case("h121_a10", 20, 10, 121, 3, "relu", ens=2, pop=40, P=3, H=6, normalize="float32"), ("ts1", "tsinf", "shuffle")),
    (_case("h138_L4_hcproc", 18, 6, 138, 4, "leaky_relu", ens=4, elites=(0, 1, 3), pop=36, P=5, H=6, normalize="float64",
           obs_process="halfcheetah", no_delta_list=(0,)), ("ts1", "tsinf", "shuffle")),
    (_case("h155_cpproc", 4, 1, 155, 2, "silu", ens=5, elites=(4, 0, 2), pop=33, P=3, H=7, normalize="float64",
           obs_process="cartpole", reward_fn="cartpole_pets"), ("ts1", "tsinf", "shuffle")),
    (_case("h172_in47", 39, 6, 172, 3, "silu", pop=30, P=5, H=5, normalize="float64", learned_rewards=True, reward_fn=None),
     ("ts1", "tsinf", "shuffle")),
    (_case("h189_in49", 40, 7, 189, 2, "relu", ens=2, pop=40, P=4, H=6, normalize="float32"), ("ts1", "tsinf", "shuffle")),
    (_case("h238_r14", 17, 6, 238, 2, "silu", pop=30, P=3, H=5, normalize="float64"), ("ts1", "tsinf", "shuffle")),
    (_case("h31_r15", 9, 2, 31, 3, "leaky_relu", pop=39, P=4, H=6), ("ts1", "tsinf", "shuffle")),
    (_case("h239_r15", 17, 6, 239, 1, "relu", ens=2, pop=32, P=3, H=5, normalize="float32"), ("ts1", "tsinf", "shuffle")),
    (_case("h254_max", 17, 6, 254, 2, "silu", ens=2, pop=30, P=4, H=5, normalize="float64"), ("ts1", "tsinf", "shuffle")),
    (_case("h24_in254_det", 248, 6, 24, 1, "relu", ens=2, pop=30, P=3, H=5, deterministic=True),
     ("ts1", "tsinf", "shuffle")),
    (_case("h64_out128", 128, 6, 64, 2, "silu", ens=2, pop=32, P=3, H=5, normalize="float64"),
     ("ts1", "tsinf", "shuffle", "expect")),
    (_case("h88_L5_fast", 17, 6, 88, 5, "silu", ens=3, pop=45, P=4, H=6, normalize="float64"), ("ts1", "tsinf", "shuffle")),
    # L >= 5 with a termination function: judged by the discrete-reward bars
    (_case("h88_L5_hopper", 11, 3, 88, 5, "silu", ens=4, elites=(3, 1), pop=32, P=4, H=6, normalize="float64",
           learned_rewards=True, reward_fn=None, term_fn="hopper", obs0_first=1.2), ("ts1", "tsinf", "shuffle")),
    # width 512: the fp32 kernel's 32-row tile; outside the tensor-core plan
    (_case("h512_f32", 17, 6, 512, 2, "silu", ens=2, pop=30, P=3, H=5, normalize="float64"), ("ts1", "tsinf", "shuffle")),
]}

# widths the tensor-core plan rejects (16: no second N half; 255: bias columns past 256)
REJECTED = {"h16": _case("h16", 5, 2, 16, 2, "silu"), "h255": _case("h255", 17, 6, 255, 2, "silu")}

# more tiles than twice the SM count, the last one partial: the config-2 model (7 members / 5 elites, 4 x 200 SiLU) at H 7
# ((L + 1) * H = 35 is odd: a CTA's next tile starts on the other activation buffer), and a hid % 16 == 8, L = 5 model
MULTI_TILE = {
    "config2_H7": (dataclasses.replace(syn.CASES["halfcheetah"], population=2000, horizon=7, particles=20), ("tsinf", "shuffle")),
    "h72_L5": (_case("mt_h72_L5", 17, 6, 72, 5, "silu", ens=5, elites=(0, 1, 2, 3), pop=2000, P=20, H=6, normalize="float64"),
               ("tsinf", "shuffle")),
    "expect_h40": (_case("mt_expect_h40", 11, 3, 40, 2, "relu", pop=1002, P=20, H=5, normalize="float32",
                         propagation="expectation"), ("expect",)),
}

ALL_CASES = {**SWEEP, **MULTI_TILE}


def mode_spec(spec, mode):
    prop = {"ts1": "random_model", "shuffle": "random_model", "tsinf": "fixed_model", "expect": "expectation"}[mode]
    return dataclasses.replace(spec, propagation=prop)


def discrete(spec):
    return spec.term_fn != "no_termination"


def _params(table):
    out = []
    for name, (spec, modes) in table.items():
        for mode in modes:
            for prec in ("f32", "bf16_tc"):
                if prec == "bf16_tc" and tc_plan(mode_spec(spec, mode), expectation=mode == "expect") is None:
                    continue
                out.append(pytest.param(name, mode, prec, id=f"{name}-{mode}-{prec}"))
    return out


# ---- GPU side -----------------------------------------------------------------------------------------------------------
class _Box:
    def __init__(self, lo, hi, n):
        self.low, self.high, self.shape = np.full(n, lo, np.float32), np.full(n, hi, np.float32), (n,)


def make_env(spec, arrays, precision, ts1):
    import mbrl_lib_b200 as bp
    from mbrl_lib_b200 import functions

    class _Env:
        observation_space = _Box(-np.inf, np.inf, spec.obs_dim)
        action_space = _Box(spec.action_lb, spec.action_ub, spec.act_dim)

    model = bp.model_from_arrays(spec, arrays, DEV)
    rew = functions.REWARD_FNS[spec.reward_fn] if spec.reward_fn else None
    env = bp.ModelEnv(_Env(), model, functions.TERM_FNS[spec.term_fn], rew, generator=torch.Generator(device=DEV),
                      precision=precision, ts1=ts1)
    env._few_groups = lambda *a: False  # tile shuffle: always the in-kernel member draw, also for these small batches
    return env


def run_case(spec, mode, precision):
    """(kernel returns, float64 oracle returns) for one case / mode / kernel."""
    from oracle import pets_oracle as po

    spec = mode_spec(spec, mode)
    arrays = syn.make_model_arrays(spec)
    inp = syn.make_rollout_inputs(spec)
    env = make_env(spec, arrays, precision, "tile_shuffle" if mode == "shuffle" else "perms")
    assert env.precision == precision
    acts = torch.from_numpy(inp["actions"])
    eps = None if spec.deterministic else torch.from_numpy(inp["eps"])
    perms = torch.from_numpy(inp["perms"]) if mode in ("ts1", "tsinf") else None
    offset = 13 * 1024
    got = env.evaluate_action_sequences(acts.to(DEV), inp["obs0"], spec.particles,
                                        _perms=None if perms is None else perms.to(DEV),
                                        _eps=None if eps is None else eps.to(DEV), _offset=offset)
    torch.cuda.synchronize()
    got = got.cpu().numpy().astype(np.float64)
    assign = None
    if mode == "shuffle":
        assign = env.shuffle_member_assignment(spec.population, spec.horizon, spec.particles, offset)
    oracle = po.OracleModel(spec, arrays, dtype=torch.float64)
    oracle.emulate_bf16 = precision == "bf16_tc"
    ref = oracle.evaluate_action_sequences(acts, inp["obs0"], spec.particles, perms, eps, assign=assign).numpy()
    return got, ref


def check(name, mode, precision, got, ref, spec):
    assert np.isfinite(got).all()
    diff = np.abs(got - ref)
    scale = max(1.0, float(np.abs(ref).max()))
    if not discrete(spec):
        tol = 2e-4 if precision == "f32" else 5e-3
        print(f"DEVIATION {name:<18} {mode:<8} {precision:<8} max|diff|/scale = {diff.max() / scale:.3e}  (bar {tol:.0e})")
        assert diff.max() <= tol * scale, f"max |diff| {diff.max():.3e} > {tol:.0e} * {scale:.3g}"
        return
    # discrete rewards (tests/test_gpu_parity.py): a particle near a termination threshold may flip
    if precision == "f32":
        bad = diff > 2e-4 * np.maximum(1.0, np.abs(ref))
        frac_bar, mean_bar = 0.02, 0.01
    else:
        bad = diff > 1e-2 * np.maximum(1.0, np.abs(ref))
        frac_bar, mean_bar = 0.01, 1e-4
    mscale = max(1.0, float(np.abs(ref).mean()))
    print(f"DEVIATION {name:<18} {mode:<8} {precision:<8} frac differing = {bad.mean():.4f} (bar {frac_bar}), "
          f"mean|diff|/scale = {diff.mean() / mscale:.3e} (bar {mean_bar:.0e}), max|diff|/scale = {diff.max() / scale:.3e}")
    assert bad.mean() <= frac_bar, f"{bad.sum()} of {bad.size} sequences differ"
    assert diff.mean() <= mean_bar * mscale, diff.mean()


@pytest.mark.gpu
@pytest.mark.parametrize("name,mode,precision", _params(SWEEP))
def test_shape_sweep_matches_float64_oracle(name, mode, precision):
    spec, _ = SWEEP[name]
    got, ref = run_case(spec, mode, precision)
    check(name, mode, precision, got, ref, spec)


@pytest.mark.gpu
@pytest.mark.parametrize("name,mode,precision", _params(MULTI_TILE))
def test_multi_tile_per_cta_matches_float64_oracle(name, mode, precision):
    from mbrl_lib_b200 import _lib

    spec, _ = MULTI_TILE[name]
    sm = C.c_int32()
    _lib.check(_lib.load().b200pets_device_info(C.byref(sm), C.byref(C.c_int32()), C.byref(C.c_int32())))
    tiles = tc_tiles(mode_spec(spec, mode), mode)
    # every CTA walks two or more tiles (one more than the SMs for "expectation"), and the last tile is partial
    assert tiles >= (sm.value + 1 if mode == "expect" else 2 * sm.value), (tiles, sm.value)
    got, ref = run_case(spec, mode, precision)
    check(name, mode, precision, got, ref, spec)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(ALL_CASES) + sorted(REJECTED))
def test_plan_restatement_matches_library(name):
    """The Python restatement of the plan (which the CPU coverage guard relies on) agrees with the library: precision
    'auto' picks the tensor-core kernel exactly for the shapes tc_plan accepts."""
    spec = ALL_CASES[name][0] if name in ALL_CASES else REJECTED[name]
    env = make_env(spec, syn.make_model_arrays(spec), "auto", "perms")
    assert env.staged.supports_tc() == (tc_plan(spec) is not None)
    assert env.precision == ("bf16_tc" if tc_plan(spec) is not None else "f32")


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(REJECTED))
def test_rejected_widths_use_fp32_path(name):
    """hid 16 and 255 are outside the tensor-core plan: 'auto' runs the fp32 kernel (and matches the oracle), asking for
    the tensor-core kernel raises instead of falling back."""
    spec = REJECTED[name]
    assert tc_plan(spec) is None
    got, ref = run_case(spec, "ts1", "f32")
    check(name, "ts1", "f32", got, ref, spec)
    arrays = syn.make_model_arrays(spec)
    env = make_env(spec, arrays, "auto", "perms")
    assert env.precision == "f32" and not env.staged.supports_tc()
    env_tc = make_env(spec, arrays, "bf16_tc", "perms")
    inp = syn.make_rollout_inputs(spec)
    with pytest.raises(NotImplementedError):
        env_tc.evaluate_action_sequences(torch.from_numpy(inp["actions"]).to(DEV), inp["obs0"], spec.particles,
                                         _perms=torch.from_numpy(inp["perms"]).to(DEV), _eps=torch.from_numpy(inp["eps"]).to(DEV))
