"""CPU oracle for the PETS planning hot path -- TEST INFRASTRUCTURE ONLY.

This is a restatement (torch CPU ops, fp32 -- or fp64 on request --, all randomness *injected*) of what the reference computes on
the path  CEMOptimizer/ICEMOptimizer -> ModelEnv.evaluate_action_sequences -> OneDTransitionRewardModel
-> GaussianMLP.  It is the checker for the CUDA path; nothing in the product imports it.  Only
``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl reference`` legs may.

Pinned: ``oracle/gen_golden.py`` drives the *imported* reference (``/root/reference`` + API shims) with
the same injected noise and stores its outputs under ``tests/golden``; ``tests/test_oracle_golden.py``
checks this file against them (bit-exact in the build container).

Reference lines each function follows are cited per function (paths relative to /root/reference).
"""
from __future__ import annotations

import math
from typing import Callable, Dict, Optional, Tuple

import numpy as np
import torch
import torch.nn.functional as F

# --------------------------------------------------------------------------------------------------
# reward / termination / observation pre-processing (mbrl/env/reward_fns.py, termination_fns.py)
# --------------------------------------------------------------------------------------------------


def term_no_termination(act, nobs):  # termination_fns.py:58-63
    return torch.zeros(nobs.shape[0], 1, dtype=torch.bool)


def term_cartpole(act, nobs):  # termination_fns.py:29-44
    x, th = nobs[:, 0], nobs[:, 2]
    lim = 12 * 2 * math.pi / 360
    ok = (x > -2.4) & (x < 2.4) & (th > -lim) & (th < lim)
    return (~ok)[:, None]


def term_inverted_pendulum(act, nobs):  # termination_fns.py:47-55
    ok = torch.isfinite(nobs).all(-1) & (nobs[:, 1].abs() <= 0.2)
    return (~ok)[:, None]


def term_hopper(act, nobs):  # termination_fns.py:12-26
    ok = (torch.isfinite(nobs).all(-1) & (nobs[:, 1:].abs() < 100).all(-1)
          & (nobs[:, 0] > 0.7) & (nobs[:, 1].abs() < 0.2))
    return (~ok)[:, None]


def term_walker2d(act, nobs):  # termination_fns.py:66-74
    h, a = nobs[:, 0], nobs[:, 1]
    ok = (h > 0.8) & (h < 2.0) & (a > -1.0) & (a < 1.0)
    return (~ok)[:, None]


def term_ant(act, nobs):  # termination_fns.py:77-85
    x = nobs[:, 0]
    ok = torch.isfinite(nobs).all(-1) & (x >= 0.2) & (x <= 1.0)
    return (~ok)[:, None]


def term_humanoid(act, nobs):  # termination_fns.py:88-95
    z = nobs[:, 0]
    return ((z < 1.0) | (z > 2.0))[:, None]


TERM_FNS: Dict[str, Callable] = {
    "no_termination": term_no_termination, "cartpole": term_cartpole,
    "inverted_pendulum": term_inverted_pendulum, "hopper": term_hopper,
    "walker2d": term_walker2d, "ant": term_ant, "humanoid": term_humanoid,
}


def rew_cartpole(act, nobs):  # reward_fns.py:10-13
    return (~term_cartpole(act, nobs)).float().view(-1, 1)


def rew_inverted_pendulum(act, nobs):  # reward_fns.py:27-30
    return (~term_inverted_pendulum(act, nobs)).float().view(-1, 1)


def rew_cartpole_pets(act, nobs):  # reward_fns.py:16-24
    goal = torch.tensor([0.0, 0.6])
    x0, th = nobs[:, :1], nobs[:, 1:2]
    ee = torch.cat([x0 - 0.6 * th.sin(), -0.6 * th.cos()], dim=1)
    obs_cost = torch.exp(-torch.sum((ee - goal) ** 2, dim=1) / (0.6 ** 2))
    act_cost = -0.01 * torch.sum(act ** 2, dim=1)
    return (obs_cost + act_cost).view(-1, 1)


def rew_halfcheetah(act, nobs):  # reward_fns.py:33-38
    ctrl = -0.1 * act.square().sum(dim=1)
    run = nobs[:, 0] - 0.0 * nobs[:, 2].square()
    return (run + ctrl).view(-1, 1)


def rew_pusher(act, nobs):  # reward_fns.py:41-53
    goal = torch.tensor([0.45, -0.05, -0.323])
    tip, obj = nobs[:, 14:17], nobs[:, 17:20]
    obs_cost = 0.5 * (tip - obj).abs().sum(dim=1) + 1.25 * (goal - obj).abs().sum(dim=1)
    act_cost = 0.1 * (act ** 2).sum(dim=1)
    return -(obs_cost + act_cost).view(-1, 1)


REWARD_FNS: Dict[str, Callable] = {
    "cartpole": rew_cartpole, "cartpole_pets": rew_cartpole_pets, "inverted_pendulum": rew_inverted_pendulum,
    "halfcheetah": rew_halfcheetah, "pusher": rew_pusher,
}


def proc_halfcheetah(s):  # mbrl/env/pets_halfcheetah.py:91-113: [o1, sin o2, cos o2, o3:]
    return torch.cat([s[..., 1:2], torch.sin(s[..., 2:3]), torch.cos(s[..., 2:3]), s[..., 3:]], dim=-1)


def proc_cartpole(s):  # mbrl/env/pets_cartpole.py:78-101: [sin o1, cos o1, o0, o2:]
    return torch.cat([torch.sin(s[..., 1:2]), torch.cos(s[..., 1:2]), s[..., :1], s[..., 2:]], dim=-1)


OBS_PROCESS: Dict[str, Callable] = {"halfcheetah": proc_halfcheetah, "cartpole": proc_cartpole}

# --------------------------------------------------------------------------------------------------
# model
# --------------------------------------------------------------------------------------------------


def _bf16_round(x: torch.Tensor) -> torch.Tensor:
    """round to bf16 and back to the working dtype (the products and sums stay in that dtype)."""
    return x.to(torch.bfloat16).to(x.dtype)


def _bf16_split_bias(b: torch.Tensor) -> torch.Tensor:
    """bias as carried by the tensor-core path: hi + lo bf16 parts (two constant-one K columns)."""
    hi = _bf16_round(b)
    return hi + _bf16_round(b - hi)


class OracleModel:
    """GaussianMLP ensemble wrapped as a OneDTransitionRewardModel, inference only.

    ``dtype=torch.float64`` runs the whole path (model input, layers, sampling, delta targets, rewards, accumulation) in
    double: the high-precision yardstick the kernels' error is measured against.  The float32 default is the reference's
    own arithmetic, pinned bit-exact to the goldens."""

    def __init__(self, spec, arrays, dtype=torch.float32):
        self.spec = spec
        self.dtype = dtype
        cast = lambda a: torch.from_numpy(np.asarray(a)).to(dtype)  # noqa: E731 (a no-op for the float32 arrays in fp32 mode)
        self.weights = [cast(w) for w in arrays["weights"]]
        self.biases = [cast(b) for b in arrays["biases"]]
        self.min_logvar = cast(arrays["min_logvar"])
        self.max_logvar = cast(arrays["max_logvar"])
        # the normaliser keeps its own dtype in fp32 mode (an fp64 normaliser promotes, then .float(), as the reference)
        self.norm_mean = self.norm_std = None
        if "norm_mean" in arrays:
            self.norm_mean = torch.from_numpy(arrays["norm_mean"])
            self.norm_std = torch.from_numpy(arrays["norm_std"])
            if dtype == torch.float64:
                self.norm_mean, self.norm_std = self.norm_mean.double(), self.norm_std.double()
        # gaussian_mlp.py:377-379: set_elite ignores a list that names as many members as the ensemble has (whatever its
        # order): all members then run in index order
        elites = spec.elites if spec.elites is not None and len(spec.elites) != spec.ensemble_size else None
        self.members = list(elites) if elites is not None else list(range(spec.ensemble_size))
        self.emulate_bf16 = False

    # mbrl/models/gaussian_mlp.py:89-111 (activation choice), models/util.py:53-65 (layer)
    def _act(self, x):
        a = self.spec.activation
        if a == "relu":
            return F.relu(x)
        if a == "silu":
            return F.silu(x)
        if a == "leaky_relu":
            return F.leaky_relu(x, 0.01)
        raise ValueError(a)

    def mlp(self, xs: torch.Tensor) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
        """xs [M, Bm, in] -> mean, logvar [M, Bm, out]   (gaussian_mlp.py:140-154)."""
        idx = self.members
        h = xs
        nl = len(self.weights)
        for li in range(nl):
            w, b = self.weights[li][idx, ...], self.biases[li][idx, ...]
            if self.emulate_bf16:
                h = _bf16_round(h).matmul(_bf16_round(w)) + _bf16_split_bias(b)
            else:
                h = h.matmul(w) + b
            if li < nl - 1:
                h = self._act(h)
        if self.spec.deterministic:
            return h, None
        out = self.spec.out_size
        mean, lv = h[..., :out], h[..., out:]
        lv = self.max_logvar - F.softplus(self.max_logvar - lv)
        lv = self.min_logvar + F.softplus(lv - self.min_logvar)
        return mean, lv

    def model_input(self, obs: torch.Tensor, act: torch.Tensor) -> torch.Tensor:
        """one_dim_tr_model.py:103-116 + util/math.py:129-143."""
        if self.spec.obs_process:
            obs = OBS_PROCESS[self.spec.obs_process](obs)
        x = torch.cat([obs, act], dim=obs.ndim - 1)
        if self.norm_mean is not None:
            x = ((x - self.norm_mean) / self.norm_std).to(self.dtype)
        return x

    def forward_assigned(self, x: torch.Tensor, assign: torch.Tensor):
        """gaussian_mlp.py:202-212 with the row -> member map given directly instead of through a permutation
        (``assign[r]`` = position in the elite list of the member row r uses).  This is what the reference computes
        for ANY permutation that induces this map; the CUDA path's in-kernel "tile shuffle" exports its map
        (b200pets_shuffle_member_map) and is checked against this function."""
        B = x.shape[0]
        M = len(self.members)
        mean_out = None
        lv_out = None
        for mpos in range(M):
            rows = torch.nonzero(assign == mpos).view(-1)
            if rows.numel() == 0:
                continue
            keep = self.members
            self.members = [keep[mpos]]
            try:
                mean, lv = self.mlp(x[rows].unsqueeze(0))
            finally:
                self.members = keep
            if mean_out is None:
                mean_out = torch.empty(B, mean.shape[-1], dtype=mean.dtype)
                lv_out = torch.empty(B, lv.shape[-1], dtype=lv.dtype) if lv is not None else None
            mean_out[rows] = mean[0]
            if lv is not None:
                lv_out[rows] = lv[0]
        return mean_out, lv_out

    def forward_propagated(self, x: torch.Tensor, perm: Optional[torch.Tensor], assign: Optional[torch.Tensor] = None):
        """gaussian_mlp.py:156-216: shuffle rows to members, run, un-shuffle (or member average)."""
        B = x.shape[0]
        M = len(self.members)
        if B % M != 0:
            raise ValueError(f"batch {B} not a multiple of {M} models")  # gaussian_mlp.py:195-200
        if assign is not None and self.spec.propagation != "expectation":
            return self.forward_assigned(x, assign)
        if self.spec.propagation == "expectation":
            mean, lv = self.mlp(x.unsqueeze(0))
            return mean.mean(dim=0), (lv.mean(dim=0) if lv is not None else None)
        xs = x[perm, ...].view(M, B // M, -1)
        mean, lv = self.mlp(xs)
        mean = mean.reshape(B, -1)
        out_mean = torch.empty_like(mean)
        out_mean[perm] = mean
        out_lv = None
        if lv is not None:
            lv = lv.reshape(B, -1)
            out_lv = torch.empty_like(lv)
            out_lv[perm] = lv
        return out_mean, out_lv

    def step(self, obs, act, perm, eps, sample=True, assign=None):
        """ModelEnv.step (model_env.py:87-140) over OneDTransitionRewardModel.sample (one_dim_tr_model.py
        :245-289) and Ensemble.sample_1d (model.py:426-473).  Returns next_obs, reward[B,1], done[B,1]."""
        sp = self.spec
        obs, act = obs.to(self.dtype), act.to(self.dtype)
        x = self.model_input(obs, act)
        mean, lv = self.forward_propagated(x, perm, assign)
        if sp.deterministic or not sample:
            preds = mean
        else:
            std = torch.sqrt(lv.exp())
            preds = mean + std * eps  # == torch.normal(mean, std, generator) for the same N(0,1) draws
        nobs = preds[:, :-1] if sp.learned_rewards else preds
        if sp.target_is_delta:
            tmp = nobs + obs
            for d in sp.no_delta_list:
                tmp[:, d] = nobs[:, d]
            nobs = tmp
        # model_env.py:124-128: `pred_rewards if self.reward_fn is None else self.reward_fn(...)`: an explicit
        # reward_fn wins even when the model also learns a reward column
        rew = REWARD_FNS[sp.reward_fn](act, nobs) if sp.reward_fn else preds[:, -1:]
        done = TERM_FNS[sp.term_fn](act, nobs)
        return nobs, rew, done

    def evaluate_action_sequences(self, actions, obs0, particles, perms, eps, return_rows=False, assign=None):
        """model_env.py:145-191.  actions [N,H,A] f32; obs0 [D]; perms [H or 1, B]; eps [H,B,out];
        assign [H or 1, B] optional row -> member map used instead of perms (see forward_assigned)."""
        N, H, _ = actions.shape
        P = particles
        B = N * P
        obs = torch.from_numpy(np.tile(np.asarray(obs0), (B, 1)).astype(np.float32)).to(self.dtype)
        total = torch.zeros(B, 1, dtype=self.dtype)
        dead = torch.zeros(B, 1, dtype=torch.bool)
        for t in range(H):
            a = torch.repeat_interleave(actions[:, t, :], P, dim=0)
            perm = None
            if self.spec.propagation != "expectation" and assign is None:
                perm = perms[0] if self.spec.propagation == "fixed_model" else perms[t]
            e = eps[t] if eps is not None else None
            asg = None
            if assign is not None:
                asg = assign[0] if assign.shape[0] == 1 else assign[t]
                perm = None
            obs, rew, done = self.step(obs, a, perm, e, sample=True, assign=asg)
            rew = rew.clone()
            rew[dead] = 0
            dead |= done
            total += rew
        if return_rows:
            return total.view(-1)
        return total.reshape(-1, P).mean(dim=1)


def mbpo_rollout(model: "OracleModel", initial_obs, policy, rollout_horizon, perms, eps, assigns=None):
    """rollout_model_and_populate_sac_buffer (mbrl/algorithms/mbpo.py:31-63) with the model noise injected: returns the
    list of per-step ``add_batch`` argument tuples (obs, action, next_obs, reward, done) -- the rows ``~accum_dones`` --
    plus the full per-step arrays for diagnostics.  ``policy(obs) -> action`` stands for ``agent.act(..., batched=True)``;
    perms[i] / eps[i] (or assigns[i]) are the draws of step i (ModelEnv.step with sample=True)."""
    obs = torch.as_tensor(np.asarray(initial_obs, dtype=np.float32))
    accum = torch.zeros(obs.shape[0], dtype=torch.bool)
    batches, full = [], []
    for i in range(rollout_horizon):
        action = policy(obs)
        nobs, rew, done = model.step(obs, action, None if perms is None else perms[i], eps[i], sample=True,
                                     assign=None if assigns is None else assigns[i])
        keep = ~accum
        batches.append((obs[keep].numpy(), action[keep].numpy(), nobs[keep].numpy(), rew[keep, 0].numpy(),
                        done[keep, 0].numpy()))
        full.append((nobs.numpy(), rew[:, 0].numpy(), done[:, 0].numpy(), keep.numpy()))
        obs = nobs
        accum = accum | done[:, 0]
    return batches, full


# --------------------------------------------------------------------------------------------------
# optimisers (mbrl/planning/trajectory_opt.py)
# --------------------------------------------------------------------------------------------------


def cem_optimize(obj_fun, x0, lb, ub, num_iterations, elite_ratio, population_size, alpha, noise,
                 return_mean_elites=False, clipped_normal=False, trace=None):
    """CEMOptimizer.optimize (trajectory_opt.py:100-188).  ``noise[i]`` [N,H,A] replaces the RNG of
    iteration i: already-truncated N(0,1) draws (truncated normal) or plain N(0,1) (clipped normal)."""
    elite_num = int(np.ceil(population_size * elite_ratio).astype(np.int32))
    mu = x0.clone()
    disp = torch.ones_like(mu) if clipped_normal else ((ub - lb) ** 2) / 16
    best_sol = torch.empty_like(mu)
    best_val = -np.inf
    for i in range(num_iterations):
        if clipped_normal:
            pop = mu + disp * noise[i]
            pop = torch.where(pop > lb, pop, lb)
            pop = torch.where(pop < ub, pop, ub)
        else:
            mv = torch.min(torch.square((mu - lb) / 2), torch.square((ub - mu) / 2))
            cvar = torch.min(mv, disp)
            pop = noise[i] * torch.sqrt(cvar) + mu
        vals = obj_fun(pop, i)
        vals = vals.clone()
        vals[vals.isnan()] = -1e-10
        bv, idx = vals.topk(elite_num)
        elite = pop[idx]
        new_mu = torch.mean(elite, dim=0)
        new_disp = torch.std(elite, dim=0) if clipped_normal else torch.var(elite, dim=0)
        mu = alpha * mu + (1 - alpha) * new_mu
        disp = alpha * disp + (1 - alpha) * new_disp
        if bv[0] > best_val:
            best_val = bv[0]
            best_sol = pop[idx[0]].clone()
        if trace is not None:
            trace.append({"pop": pop, "values": vals, "elite_idx": idx, "mu": mu.clone(), "disp": disp.clone()})
    return mu if return_mean_elites else best_sol


def powerlaw_psd_from_normals(exponent, sr, si, samples):
    """util/math.py:318-396 with the two N(0,1) draws injected: sr, si [..., samples//2+1] (unit normals,
    scaled here by the spectrum).  Returns [..., samples]."""
    f = torch.fft.rfftfreq(samples)
    s_scale = f.clone()
    fmin = max(0.0, 1.0 / samples)
    ix = int(torch.sum(s_scale < fmin))
    if ix and ix < len(s_scale):
        s_scale[:ix] = s_scale[ix]
    s_scale = s_scale ** (-exponent / 2.0)
    w = s_scale[1:].detach().clone()
    w[-1] *= (1 + (samples % 2)) / 2.0
    sigma = 2 * torch.sqrt(torch.sum(w ** 2)) / samples
    sr = sr * s_scale
    si = si * s_scale
    si = si.clone()
    if not (samples % 2):
        si[..., -1] = 0
    si[..., 0] = 0
    return torch.fft.irfft(sr + 1j * si, n=samples, dim=-1) / sigma


def icem_population_sizes(num_iterations, population_size, decay, elite_num, module=None):
    """trajectory_opt.py:410-431."""
    out = []
    for i in range(num_iterations):
        n = int(np.ceil(np.max((population_size * decay ** -i, 2 * elite_num))).astype(np.int32))
        if module and n % module:
            n += module - n % module
        out.append(n)
    return out


def icem_optimize(obj_fun, x0, lb, ub, num_iterations, elite_ratio, population_size, decay, exponent,
                  keep_elite_frac, alpha, noise, prev_elite=None, return_mean_elites=False, module=None, trace=None):
    """ICEMOptimizer.optimize (trajectory_opt.py:391-487).  ``noise[i]`` is a dict with the injected draws of
    iteration i: 'sr','si' [n_i, A, H//2+1]; 'keep_perm' [elite_num] (if an elite set exists);
    'end_eps' [keep, A] (iteration 0 with previous elites).  Returns (solution, elite set)."""
    elite_num = int(np.ceil(population_size * elite_ratio).astype(np.int32))
    keep = int(np.ceil(keep_elite_frac * elite_num).astype(np.int32))
    if module and keep % module:
        keep += module - keep % module
    H, A = x0.shape
    mu = x0.clone()
    var = (((ub - lb) ** 2) / 16).clone()
    best_sol = torch.empty_like(mu)
    best_val = -np.inf
    elite = prev_elite
    sizes = icem_population_sizes(num_iterations, population_size, decay, elite_num, module)
    for i in range(num_iterations):
        nz = noise[i]
        colored = powerlaw_psd_from_normals(exponent, nz["sr"], nz["si"], H).transpose(1, 2)
        assert colored.shape[0] == sizes[i]
        pop = torch.minimum(colored * torch.sqrt(var) + mu, ub)
        pop = torch.maximum(pop, lb)
        if elite is not None:
            kept = torch.index_select(elite, 0, nz["keep_perm"][:keep])
            if i == 0:
                end = (mu[-1, :].repeat(kept.shape[0], 1)
                       + torch.sqrt(var[-1, :]).repeat(kept.shape[0], 1) * nz["end_eps"]).unsqueeze(1)
                pop = torch.cat((pop, torch.cat((kept[:, 1:, :], end), dim=1)), dim=0)
            elif i == num_iterations - 1:
                pop = torch.cat((pop, mu.unsqueeze(0)), dim=0)
            else:
                pop = torch.cat((pop, kept), dim=0)
        vals = obj_fun(pop, i).clone()
        vals[vals.isnan()] = -1e-10
        bv, idx = vals.topk(elite_num)
        elite = pop[idx]
        mu = alpha * mu + (1 - alpha) * torch.mean(elite, dim=0)
        var = alpha * var + (1 - alpha) * torch.var(elite, unbiased=False, dim=0)
        if bv[0] > best_val:
            best_val = bv[0]
            best_sol = pop[idx[0]].clone()
        if trace is not None:
            trace.append({"pop": pop, "values": vals, "elite_idx": idx, "mu": mu.clone(), "var": var.clone()})
    return (mu if return_mean_elites else best_sol), elite


def mppi_optimize(obj_fun, mean, lb, ub, num_iterations, population_size, gamma, beta, noise, trace=None):
    """MPPIOptimizer.optimize (trajectory_opt.py:233-311).  ``mean`` [H,A] is the optimiser's state (returned updated);
    ``noise[k]`` [N,H,A] are the (already truncated) N(0,1) draws of refinement k.  Note two quirks restated as is:
    ``past_action`` aliases mean[0] and therefore holds the *shifted* row, and the variance-scaled population is
    overwritten by mean + unscaled noise."""
    mean = mean.clone()
    mean[:-1] = mean[1:].clone()
    past_action = mean[0].clone()
    H = mean.shape[0]
    for k in range(num_iterations):
        nz = noise[k]
        pop = torch.empty_like(nz)
        pop[:, 0, :] = beta * (mean[0, :] + nz[:, 0, :]) + (1 - beta) * past_action
        for i in range(max(H - 1, 0)):
            pop[:, i + 1, :] = beta * (mean[i + 1] + nz[:, i + 1, :]) + (1 - beta) * pop[:, i, :]
        pop = torch.where(pop > ub, ub, pop)
        pop = torch.where(pop < lb, lb, pop)
        vals = obj_fun(pop, k).clone()
        vals[vals.isnan()] = -1e-10
        w = torch.reshape(torch.exp(gamma * (vals - vals.max())), (population_size, 1, 1))
        norm = torch.sum(w) + 1e-10
        mean = torch.sum(pop * w, dim=0) / norm
        if trace is not None:
            trace.append({"pop": pop, "values": vals, "mean": mean.clone()})
    return mean


def shift_solution(best, replan_freq, initial_row):
    """TrajectoryOptimizer.optimize warm start (trajectory_opt.py:563-567)."""
    prev = best.roll(-replan_freq, dims=0)
    prev[-replan_freq:] = initial_row
    return prev
