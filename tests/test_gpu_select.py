"""Elite selection + refit (csrc/cem.cu, b200pets_cem_update) on each of its three code paths, against a float64 NumPy
restatement of the rule:

  * NaN -> -1e-10f, in place (trajectory_opt.py:178);
  * the k largest values, ties at the k-th position to the lowest population index, -0.0 == +0.0 (a tie, not an order);
  * ``elite_idx`` ascending; ``elites_out`` rows by descending value, ties by lower index (the order of topk's rows);
  * mean and (un)biased variance -- or its square root -- over the elites, momentum ``alpha``;
  * best-so-far: the maximum value, lowest index on ties, replaces ``best`` only when strictly larger.

Paths (run_select in cem.cu):
  small   n <= 2048 and k * dims * 4 <= 150 KB   cem_select_small_kernel: counting rank, elites staged in shared memory
  count   n <= 2048, elites do not fit           cem_select_kernel: counting rank, global reads (config 3's iCEM shape)
  radix   n > 2048                               cem_select_kernel: 4-pass radix select on the order-preserving key
The peer-exchange kernel of the sharded CEM (cem_elites_refit_sample_kernel) runs the same radix select; its world = 1
form is checked on the +-0 case.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from mbrl_lib_b200 import _lib

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SMALL_SMEM = 150 * 1024  # elite rows the small-population kernel stages in shared memory


def path_of(n, k, dims):
    if n > 2048:
        return "radix"
    return "small" if k * dims * 4 <= SMALL_SMEM else "count"


# ---- the rule, in float64 ------------------------------------------------------------------------------------------
def reference_update(pop, values, mu, disp, best_v, best_s, k, alpha, unbiased, use_std):
    v = values.astype(np.float32).copy()
    v[np.isnan(v)] = np.float32(-1e-10)
    key = v.astype(np.float64) + 0.0  # -0.0 + 0.0 == +0.0: the two zeros are one key
    order = np.lexsort((np.arange(len(v)), -key))  # descending value, then ascending index
    top = order[:k]
    idx = np.sort(top)
    el = pop[idx].astype(np.float64)
    mean = el.mean(axis=0)
    var = ((el - mean) ** 2).sum(axis=0) / (k - 1 if unbiased else k)
    nd = np.sqrt(var) if use_std else var
    out = dict(values=v, elite_idx=idx, elites_out=pop[top], mu=alpha * mu.astype(np.float64) + (1 - alpha) * mean,
               disp=alpha * disp.astype(np.float64) + (1 - alpha) * nd, best_value=np.float32(best_v),
               best_solution=best_s.copy())
    if v[order[0]] > best_v:
        out["best_value"] = v[order[0]]
        out["best_solution"] = pop[order[0]].copy()
    return out


def test_reference_rule_self_check():
    """The restatement itself on a hand-checked vector (CPU arithmetic; runs with the GPU suite)."""
    v = np.array([1.0, np.nan, -1e-10, 3.0, -0.0, 0.0, 3.0, -np.inf], np.float32)
    pop = np.arange(8, dtype=np.float32)[:, None] * np.ones((1, 2), np.float32)
    r = reference_update(pop, v, np.zeros(2), np.ones(2), -np.inf, np.zeros(2), 5, 0.0, 0, 0)
    assert r["elite_idx"].tolist() == [0, 3, 4, 5, 6]        # 3, 3, 1, then the zeros (-0 at 4 ties +0 at 5)
    assert r["elites_out"][:, 0].tolist() == [3, 6, 0, 4, 5]
    r = reference_update(pop, v, np.zeros(2), np.ones(2), -np.inf, np.zeros(2), 6, 0.0, 0, 0)
    assert r["elite_idx"].tolist() == [0, 1, 3, 4, 5, 6]  # the NaN (-1e-10 at index 1) ties -1e-10 at 2: lower index
    assert r["best_value"] == 3.0 and r["best_solution"][0] == 3.0


# ---- value patterns ------------------------------------------------------------------------------------------------
def _values(kind, n, k, g):
    v = g.standard_normal(n).astype(np.float32)
    if kind == "random":
        return v
    if kind == "all_equal":
        return np.full(n, 0.25, np.float32)
    if kind == "ties_at_k":  # a run of equal values around the k-th position, interleaved with others in index order
        if n < 4:
            return np.array([0.5] * n, np.float32)
        t = np.sort(v)[::-1][min(k, n) - 1]
        ranks = np.argsort(-v, kind="stable")
        tie = ranks[max(0, k - 3):min(n, k + 3)]
        v[tie] = t
        return v
    if kind == "nan_vs_tiny":  # NaN becomes -1e-10: it ties genuine -1e-10 values; both sit at the threshold
        v = -1.0 - np.abs(v)
        pos = max(0, k - 4)
        v[g.permutation(n)[:pos]] = 1.0 + np.abs(v[:pos])
        rest = np.flatnonzero(v < 0)
        m = min(len(rest), 10)
        pick = np.sort(g.choice(rest, m, replace=False))
        v[pick[0::2]] = np.float32(-1e-10)
        v[pick[1::2]] = np.nan
        return v
    if kind == "inf":
        idx = g.permutation(n)
        v[idx[:max(1, k // 3)]] = np.inf
        v[idx[max(1, k // 3):max(1, k // 3) + max(1, n // 5)]] = -np.inf
        return v
    if kind == "signed_zero":  # -0.0 at the lower indices, +0.0 at the higher ones; the k-th value is zero
        v = -1.0 - np.abs(v)
        pos = max(0, k - 3)
        v[g.permutation(n)[:pos]] = 1.0 + np.abs(v[:pos])
        zeros = np.sort(g.choice(np.flatnonzero(v < 0), min(8, int((v < 0).sum())), replace=False))
        half = len(zeros) // 2
        v[zeros[:half]] = -0.0
        v[zeros[half:]] = 0.0
        return v
    if kind == "subnormal":
        tiny = np.array([1e-45, -1e-45, 1e-40, -1e-40, 1.2e-38, 0.0, -0.0], np.float32)
        return tiny[g.integers(0, len(tiny), n)]
    if kind == "deep_radix":  # share the top three bytes of the key: the last radix pass decides, with duplicates
        bits = np.uint32(0x3F812300) | g.integers(0, 64, n).astype(np.uint32)
        return bits.view(np.float32)
    raise ValueError(kind)


KINDS = ["random", "all_equal", "ties_at_k", "nan_vs_tiny", "inf", "signed_zero", "subnormal", "deep_radix"]


def _problem(n, dims, kind, k, seed):
    g = np.random.default_rng([n, dims, k, seed, KINDS.index(kind)])
    pop = (g.uniform(-1, 1, (n, dims)) + np.linspace(-2, 2, dims)).astype(np.float32)  # distinct rows, nonzero means
    mu = g.uniform(-0.5, 0.5, dims).astype(np.float32)
    disp = g.uniform(0.05, 0.5, dims).astype(np.float32)
    return pop, _values(kind, n, k, g), mu, disp


def cem_update(pop, values, mu, disp, best_v, best_s, k, alpha, unbiased, use_std, with_elites):
    lib = _lib.load()
    n, dims = pop.shape
    d = {name: torch.from_numpy(np.ascontiguousarray(a)).to(DEV) for name, a in
         (("pop", pop), ("val", values), ("mu", mu), ("disp", disp), ("best_s", best_s))}
    d["best_v"] = torch.tensor([best_v], dtype=torch.float32, device=DEV)
    idx = torch.full((k,), -1, dtype=torch.int32, device=DEV)
    eo = torch.full((k, dims), np.nan, device=DEV) if with_elites else None
    ws = torch.empty(lib.b200pets_cem_update_workspace_bytes(n, dims, k), dtype=torch.uint8, device=DEV)
    _lib.check(lib.b200pets_cem_update(n, dims, k, alpha, int(unbiased), int(use_std), _lib.ptr(d["pop"]), _lib.ptr(d["val"]),
                                       _lib.ptr(d["mu"]), _lib.ptr(d["disp"]), _lib.ptr(d["best_v"]), _lib.ptr(d["best_s"]),
                                       _lib.ptr(idx), _lib.ptr(eo), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
    torch.cuda.synchronize()
    return dict(values=d["val"].cpu().numpy(), elite_idx=idx.cpu().numpy(), mu=d["mu"].cpu().numpy(),
                disp=d["disp"].cpu().numpy(), best_value=d["best_v"].cpu().numpy()[0], best_solution=d["best_s"].cpu().numpy(),
                elites_out=None if eo is None else eo.cpu().numpy())


def assert_matches(got, want, where):
    np.testing.assert_array_equal(got["elite_idx"], want["elite_idx"], err_msg=f"{where}: elite_idx")
    np.testing.assert_array_equal(got["values"], want["values"], err_msg=f"{where}: values after the NaN rule")
    if got.get("elites_out") is not None:
        np.testing.assert_array_equal(got["elites_out"], want["elites_out"], err_msg=f"{where}: elites_out order")
    assert got["best_value"] == want["best_value"], f"{where}: best value {got['best_value']} != {want['best_value']}"
    np.testing.assert_array_equal(got["best_solution"], want["best_solution"], err_msg=f"{where}: best solution")
    for name in ("mu", "disp"):
        np.testing.assert_allclose(got[name], want[name], rtol=1e-5, atol=1e-7, err_msg=f"{where}: {name}")


# (unbiased, use_std): CEM's variance, the clipped-normal CEM's std, iCEM's biased variance, and the fourth combination
FLAGS = [(1, 0), (1, 1), (0, 0), (0, 1)]


def _ks(n):
    return sorted({k for k in (2, n // 10, n) if k >= 2})


SHAPES = [(n, k) for n in (2, 500, 2047, 2048, 2049, 64000) for k in _ks(n)]


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n,k", SHAPES)
def test_cem_update_matches_rule(n, k, kind):
    dims = 6
    pop, values, mu, disp = _problem(n, dims, kind, k, 0)
    best_s0 = np.full(dims, 7.0, np.float32)
    for fi, (unbiased, use_std) in enumerate(FLAGS):
        for with_elites in (False, True):
            if with_elites and k > 6400:  # elites_out ranks the k elites pairwise in one CTA: O(k^2) work
                continue
            best_v0 = -np.inf if fi % 2 == 0 else 0.5  # best-so-far replaced / kept
            want = reference_update(pop, values, mu, disp, best_v0, best_s0, k, 0.1, unbiased, use_std)
            got = cem_update(pop, values, mu, disp, best_v0, best_s0, k, 0.1, unbiased, use_std, with_elites)
            assert_matches(got, want, f"{path_of(n, k, dims)} n={n} k={k} {kind} unbiased={unbiased} std={use_std}")


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n,k,dims", [(1000, 100, 384),   # k * dims * 4 == 150 KB exactly: small path
                                      (1000, 101, 384),   # one elite row more: counting path
                                      (1000, 100, 680),   # config 3's iCEM: pop 1000, H 40 x A 17, k 100 (272 KB)
                                      (2048, 2048, 19)])  # every row an elite, above the staging limit
def test_cem_update_shared_memory_boundary(n, k, dims, kind):
    pop, values, mu, disp = _problem(n, dims, kind, k, 1)
    best_s0 = np.zeros(dims, np.float32)
    for unbiased, use_std in FLAGS:
        for with_elites in (False, True):
            want = reference_update(pop, values, mu, disp, -np.inf, best_s0, k, 0.25, unbiased, use_std)
            got = cem_update(pop, values, mu, disp, -np.inf, best_s0, k, 0.25, unbiased, use_std, with_elites)
            assert_matches(got, want, f"{path_of(n, k, dims)} n={n} k={k} dims={dims} {kind}")


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("k", [2, 100, 2000])
def test_all_three_paths_pick_the_same_elites(kind, k):
    """The same 2000 values through the small path (dims 4), the counting path (dims wide enough that the k elite rows
    exceed 150 KB) and the radix path (the values followed by 49 -inf, n = 2049: the padding never wins a tie)."""
    n = 2000
    g = np.random.default_rng([k, KINDS.index(kind), 7])
    values = _values(kind, n, k, g)
    results = {}
    for path, dims, pad in (("small", 4, 0), ("count", SMALL_SMEM // (4 * k) + 1, 0), ("radix", 4, 49)):
        v = np.concatenate([values, np.full(pad, -np.inf, np.float32)])
        pop = g.uniform(-1, 1, (n + pad, dims)).astype(np.float32)
        assert path_of(n + pad, k, dims) == path
        got = cem_update(pop, v, np.zeros(dims, np.float32), np.ones(dims, np.float32), -np.inf, np.zeros(dims, np.float32),
                         k, 0.1, 1, 0, True)
        want = reference_update(pop, v, np.zeros(dims), np.ones(dims), -np.inf, np.zeros(dims, np.float32), k, 0.1, 1, 0)
        assert_matches(got, want, f"{path} k={k} {kind}")
        results[path] = got["elite_idx"]
    assert np.array_equal(results["small"], results["count"]) and np.array_equal(results["small"], results["radix"])


@pytest.mark.parametrize("n,k", [(500, 50), (2049, 205), (40000, 4000)])  # (40 960 sequences per rank at most)
def test_signed_zero_ties_in_peer_exchange_refit(n, k):
    """The sharded CEM's select (world = 1: values push + radix select + elite table + refit) keeps the +-0 tie rule:
    its refit equals the rule's, and equals b200pets_cem_update's on the same values."""
    lib = _lib.load()
    dims = 8
    pop, values, mu, disp = _problem(n, dims, "signed_zero", k, 2)
    want = reference_update(pop, values, mu, disp, -np.inf, np.zeros(dims, np.float32), k, 0.1, 1, 0)
    single = cem_update(pop, values, mu, disp, -np.inf, np.zeros(dims, np.float32), k, 0.1, 1, 0, False)
    assert_matches(single, want, f"cem_update n={n}")
    nbytes = lib.b200pets_peer_buffer_bytes(1, n, dims, k)
    buf, handle = C.c_void_p(), C.create_string_buffer(64)
    _lib.check(lib.b200pets_peer_alloc(nbytes, C.byref(buf), handle))
    try:
        ptrs = (C.c_void_p * 1)(buf.value)
        pop_d, val_d = torch.from_numpy(pop).to(DEV), torch.from_numpy(values.copy()).to(DEV)
        mu_d, disp_d = torch.from_numpy(mu).to(DEV), torch.from_numpy(disp).to(DEV)
        best_v = torch.full((1,), float("-inf"), device=DEV)
        best_s = torch.zeros(dims, device=DEV)
        tag = torch.zeros(1, dtype=torch.int32, device=DEV)
        _lib.check(lib.b200pets_cem_values_push(n, dims, k, _lib.ptr(val_d), 0, 1, 1, ptrs, _lib.stream_ptr()))
        _lib.check(lib.b200pets_cem_elites_refit(n, 0, dims, k, 0.1, 0, 0, 1, 1, ptrs, _lib.ptr(pop_d), _lib.ptr(mu_d),
                                                 _lib.ptr(disp_d), _lib.ptr(best_v), _lib.ptr(best_s), 0, None, None, 0, 0, 0,
                                                 _lib.ptr(tag), None, _lib.stream_ptr()))
        torch.cuda.synchronize()
        got = dict(mu=mu_d.cpu().numpy(), disp=disp_d.cpu().numpy())
        for name in ("mu", "disp"):
            np.testing.assert_allclose(got[name], want[name], rtol=1e-5, atol=1e-7, err_msg=f"peer exchange n={n}: {name}")
        assert best_v.item() == want["best_value"]
        np.testing.assert_array_equal(best_s.cpu().numpy(), want["best_solution"])
    finally:
        lib.b200pets_peer_close(buf, 1)
