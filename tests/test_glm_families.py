"""GLM families with fitted parameters (normal, Student-t, negative binomial): the fp64 oracle, the
[intercept, beta, phi] layout through every Python layer, and input validation (CPU, collective backend)."""
import asyncio
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.stats
import torch

from pytensor_federated_b200.batching import DynamicBatcher, stacked_compute_func
from pytensor_federated_b200.federation import NodeFederation
from pytensor_federated_b200.models import FAMILY_PARAMS, Fp8GlmShards, GlmShards, synth_glm_shard
from pytensor_federated_b200.parallel import FederatedEngine
from pytensor_federated_b200.parallel.engine import default_inputs_from_words
from pytensor_federated_b200.sampling import glm_batch_fn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAMILIES = ["normal", "student_t", "negative_binomial"]
PHI = {"normal": [0.7], "student_t": [1.3, 4.5], "negative_binomial": [2.5]}
DATA_PHI = {"normal": (0.7,), "student_t": (1.3, 4.0), "negative_binomial": (2.0,)}
P = 8


def _data(family, rows=(230, 97), seed=0):
    Xs, ys = [], []
    for i, n in enumerate(rows):
        X, y, _ = synth_glm_shard(n, P, family=family, phi=DATA_PHI[family], seed=seed + i, device="cpu",
                                  beta_scale=0.3, intercept=1.0)
        Xs.append(X)
        ys.append(y)
    return Xs, ys


def _inputs(K=1, seed=1, D=1):
    rng = np.random.default_rng(seed)
    if K == 1:
        return rng.normal(size=2) * 0.2 + 0.8, rng.normal(size=P) * 0.2
    return rng.normal(size=(K, 2)) * 0.2 + 0.8, rng.normal(size=(K, P)) * 0.2


def _scipy_logp(family, Xs, ys, groups, ic, beta, phi):
    total = 0.0
    for X, y, g in zip(Xs, ys, groups):
        eta = X.double().numpy() @ beta + ic[g]
        y = y.double().numpy()
        if family == "normal":
            total += scipy.stats.norm.logpdf(y, eta, phi[0]).sum()
        elif family == "student_t":
            total += scipy.stats.t.logpdf(y, phi[1], eta, phi[0]).sum()
        else:
            mu = np.exp(eta)
            total += scipy.stats.nbinom.logpmf(y, phi[0], phi[0] / (phi[0] + mu)).sum()
    return total


@pytest.mark.parametrize("family", FAMILIES)
def test_reference_partial_equals_scipy_log_density(family):
    Xs, ys = _data(family)
    model = GlmShards(Xs, ys, groups=[0, 1], n_groups=2, family=family)
    assert model.family_param_names == FAMILY_PARAMS[family] and model.n_inputs == 3
    ic, beta = _inputs()
    phi = np.array(PHI[family])
    logp, d_ic, d_beta, d_phi = model.unpack_result(model.reference_partial([ic, beta, phi], dtype=torch.float64))
    assert d_ic.shape == (2,) and d_beta.shape == (P,) and d_phi.shape == (len(phi),)
    np.testing.assert_allclose(logp, _scipy_logp(family, Xs, ys, [0, 1], ic, beta, phi), rtol=1e-10)


def test_negative_binomial_oracle_with_large_counts_and_dispersions():
    X = torch.randn(64, P).to(torch.bfloat16)
    y = torch.tensor(np.r_[np.arange(60) * 37 % 1500, [0, 1, 2500, 1001]], dtype=torch.float32)
    model = GlmShards([X], [y], family="negative_binomial")
    for alpha in (0.5, 5.0, 500.0):
        ic, beta = np.array([5.0]), np.full(P, 0.05)
        logp = model.unpack_result(model.reference_partial([ic, beta, np.array([alpha])], dtype=torch.float64))[0]
        np.testing.assert_allclose(logp, _scipy_logp("negative_binomial", [X], [y], [0], ic, beta, [alpha]), rtol=1e-10)


@pytest.mark.parametrize("family", FAMILIES)
def test_every_gradient_block_matches_central_differences(family):
    Xs, ys = _data(family, seed=5)
    model = GlmShards(Xs, ys, groups=[0, 1], n_groups=2, family=family)
    ic, beta = _inputs(seed=2)
    phi = np.array(PHI[family])

    def f(ic, beta, phi):
        return model.unpack_result(model.reference_partial([ic, beta, phi], dtype=torch.float64))

    _, d_ic, d_beta, d_phi = f(ic, beta, phi)
    h = 1e-6
    for arr, grad, slot in ((ic, d_ic, 0), (beta, d_beta, 1), (phi, d_phi, 2)):
        for i in range(arr.size):
            plus, minus = [ic.copy(), beta.copy(), phi.copy()], [ic.copy(), beta.copy(), phi.copy()]
            plus[slot][i] += h
            minus[slot][i] -= h
            fd = (float(f(*plus)[0]) - float(f(*minus)[0])) / (2 * h)
            np.testing.assert_allclose(grad[i], fd, rtol=1e-6, atol=1e-5)


@pytest.mark.parametrize("K", [1, 3])
def test_packing_round_trips(K):
    Xs, ys = _data("student_t")
    model = GlmShards(Xs, ys, groups=[0, 1], n_groups=2, family="student_t", n_chains=K)
    assert model.n_params == 2 + P + 2 and model.n_vals == K * (1 + 2 + P + 2)
    ic, beta = _inputs(K)
    phi = np.array([[1.5, 3.0 + k] for k in range(K)]) if K > 1 else np.array([1.5, 3.0])
    words = np.zeros(model.n_theta_words, dtype=np.uint32)
    model.pack_theta([ic, beta, phi], words)
    th = words.view(np.float32).reshape(K, 2 + P + 2)
    np.testing.assert_array_equal(th[:, -2:], np.asarray(phi, np.float32).reshape(K, 2))
    back = default_inputs_from_words(model, words)
    assert len(back) == 3
    for got, want in zip(back, (ic, beta, phi)):
        np.testing.assert_array_equal(got, np.asarray(want, dtype=np.float32))
    vals = np.arange(model.n_vals, dtype=np.float64)
    logp, d_ic, d_beta, d_phi = model.unpack_result(vals, model.call_context([ic, beta, phi]))
    rows = vals.reshape(K, -1)
    np.testing.assert_array_equal(np.reshape(logp, -1), rows[:, 0])
    np.testing.assert_array_equal(np.reshape(d_ic, (K, 2)), rows[:, 1:3])
    np.testing.assert_array_equal(np.reshape(d_beta, (K, P)), rows[:, 3 : 3 + P])
    np.testing.assert_array_equal(np.reshape(d_phi, (K, 2)), rows[:, 3 + P :])


def test_collective_engine_evaluates_the_oracle_and_batches():
    Xs, ys = _data("negative_binomial")
    K = 3
    model = GlmShards(Xs, ys, groups=[0, 1], n_groups=2, family="negative_binomial", n_chains=K)
    ic, beta = _inputs(K)
    phi = np.array([[0.5], [5.0], [500.0]])
    with FederatedEngine(model, backend="collective") as eng:
        got = eng.evaluate(ic, beta, phi)
    for k in range(K):
        single = GlmShards(Xs, ys, groups=[0, 1], n_groups=2, family="negative_binomial")
        want = single.reference([ic[k], beta[k], phi[k]])
        for g, w in zip(got, want):
            np.testing.assert_allclose(np.asarray(g)[k], w, rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("family", ["normal", "negative_binomial"])
def test_node_federation_matches_single_node_engines(family):
    rows = (150, 170, 190)
    Xs, ys = _data(family, rows=rows, seed=7)
    model = GlmShards(Xs, ys, groups=[0, 1, 0], n_groups=2, n_chains=3, family=family, node_ids=[0, 1, 2], n_nodes=3)
    fed = NodeFederation(FederatedEngine(model, backend="collective"))
    ic, beta = _inputs(seed=3)
    phis = [np.array([0.8]), np.array([1.1]), np.array(2.0)]        # a scalar phi is fine for D = 1
    res = fed.evaluate_nodes({i: (ic, beta, phis[i]) for i in range(3)})
    assert fed.n_launches == 1
    for i in range(3):
        single = FederatedEngine(GlmShards([Xs[i]], [ys[i]], groups=[[0, 1, 0][i]], n_groups=2, family=family),
                                 backend="collective")
        want = single.logp_grad(ic, beta, np.atleast_1d(phis[i]))
        np.testing.assert_allclose(res[i][0], want[0], rtol=1e-6)
        for g, w in zip(res[i][1], want[1]):
            np.testing.assert_allclose(np.reshape(g, -1), np.reshape(w, -1), rtol=1e-5, atol=1e-5)
        assert np.shape(res[i][1][2]) == np.shape(phis[i])
    with pytest.raises(ValueError, match="3 inputs"):
        fed.evaluate_nodes({0: (ic, beta)})
    # the whole federation as one function of (intercept, beta, phi)
    one_chain = GlmShards(Xs, ys, groups=[0, 1, 0], n_groups=2, family=family, node_ids=[0, 1, 2], n_nodes=3)
    func = NodeFederation(FederatedEngine(one_chain, backend="collective")).all_nodes_func()
    logp, grads = func(ic, beta, np.array([0.9]))
    pooled = FederatedEngine(GlmShards(Xs, ys, groups=[0, 1, 0], n_groups=2, family=family), backend="collective")
    want = pooled.evaluate(ic, beta, np.array([0.9]))
    np.testing.assert_allclose(logp, want[0], rtol=1e-6)
    for g, w in zip(grads, want[1:]):
        np.testing.assert_allclose(g, w, rtol=1e-5, atol=1e-5)


class _Fp64Engine:
    """The engine interface glm_batch_fn uses, evaluated by the fp64 oracle without the float32 theta words
    (finite differences need the unrounded parameters)."""

    def __init__(self, model):
        self.model = model

    def evaluate(self, *inputs):
        return self.model.unpack_result(self.model.reference_partial(list(inputs), dtype=torch.float64),
                                        self.model.call_context(inputs))


def test_glm_batch_fn_works_in_log_phi_space():
    Xs, ys = _data("student_t")
    K = 2
    model = GlmShards(Xs, ys, groups=[0, 1], n_groups=2, family="student_t", n_chains=K)
    fn = glm_batch_fn(_Fp64Engine(model), 2)
    rng = np.random.default_rng(0)
    theta = np.concatenate([rng.normal(size=(3, 2)) * 0.2 + 0.8, rng.normal(size=(3, P)) * 0.2,
                            np.log([[1.2, 4.0], [0.9, 7.0], [1.5, 3.0]])], axis=1)   # 3 chains on a K = 2 engine
    lp, grad = fn(theta)
    assert lp.shape == (3,) and grad.shape == theta.shape
    one = _Fp64Engine(GlmShards(Xs, ys, groups=[0, 1], n_groups=2, family="student_t"))
    for k in range(3):
        want = float(one.evaluate(theta[k, :2], theta[k, 2:-2], np.exp(theta[k, -2:]))[0]) + theta[k, -2:].sum()
        np.testing.assert_allclose(lp[k], want, rtol=1e-12)
    h = 1e-6
    for j in (0, 3, theta.shape[1] - 2, theta.shape[1] - 1):
        tp, tm = theta.copy(), theta.copy()
        tp[:, j] += h
        tm[:, j] -= h
        fd = (fn(tp)[0] - fn(tm)[0]) / (2 * h)
        np.testing.assert_allclose(grad[:, j], fd, rtol=1e-6, atol=1e-5)
    # the collective engine (float32 theta words) agrees with the oracle path
    lp32, grad32 = glm_batch_fn(FederatedEngine(model, backend="collective"), 2)(theta)
    np.testing.assert_allclose(lp32, lp, rtol=1e-5)
    np.testing.assert_allclose(grad32, grad, rtol=1e-3, atol=1e-2)


def test_existing_families_keep_two_inputs_in_glm_batch_fn():
    X = torch.randn(100, P).to(torch.bfloat16)
    y = (torch.rand(100) < 0.5).float()
    model = GlmShards([X], [y], n_chains=2)
    assert model.n_inputs == 2 and model.n_family_params == 0 and model.family_param_names == ()
    lp, grad = glm_batch_fn(FederatedEngine(model, backend="collective"), 1)(np.zeros((2, 1 + P)))
    assert lp.shape == (2,) and grad.shape == (2, 1 + P)


def test_invalid_inputs_are_rejected():
    X = torch.randn(50, P).to(torch.bfloat16)
    with pytest.raises(ValueError, match="integer counts"):
        GlmShards([X], [torch.full((50,), 1.5)], family="negative_binomial")
    with pytest.raises(ValueError, match="integer counts"):
        GlmShards([X], [torch.full((50,), -1.0)], family="negative_binomial")
    model = GlmShards([X], [torch.arange(50.0)], family="negative_binomial")
    words = np.zeros(model.n_theta_words, dtype=np.uint32)
    for bad in (0.0, -1.0, np.nan, np.inf):
        with pytest.raises(ValueError, match="> 0"):
            model.pack_theta([np.zeros(1), np.zeros(P), np.array([bad])], words)
        with pytest.raises(ValueError, match="> 0"):
            model.reference_partial([np.zeros(1), np.zeros(P), np.array([bad])])
    assert not words.any()   # a rejected call writes nothing
    with pytest.raises(ValueError, match="3 inputs"):
        model.pack_theta([np.zeros(1), np.zeros(P)], words)
    # only the tensor-core kernel has these families; the collective backend works for any kernel= value
    for kernel in ("simt", "generic", "fp8"):
        m = GlmShards([X], [torch.arange(50.0)], family="negative_binomial", kernel=kernel)
        with pytest.raises(ValueError, match="tensor-core kernel only"):
            m.use_tensor_cores()
        with FederatedEngine(m, backend="collective") as eng:
            assert np.isfinite(eng.evaluate(np.zeros(1), np.zeros(P), np.array([2.0]))[0])
    odd = GlmShards([torch.randn(50, 12).to(torch.bfloat16)], [torch.zeros(50)], family="normal")
    with pytest.raises(ValueError, match="P % 8 == 0"):
        odd.use_tensor_cores()
    assert GlmShards([X], [torch.zeros(50)], family="normal").use_tensor_cores() == 1
    with pytest.raises(ValueError, match="fp8 kernel has no"):
        Fp8GlmShards.from_dense([torch.randn(128, 128)], [torch.arange(128.0)], family="negative_binomial")


def test_dynamic_batcher_serves_a_three_input_engine():
    Xs, ys = _data("normal")
    K = 4
    model = GlmShards(Xs, ys, groups=[0, 1], n_groups=2, family="normal", n_chains=K)
    eng = FederatedEngine(model, backend="collective")
    batcher = DynamicBatcher(stacked_compute_func(eng.evaluate, max_batch=K), max_batch=K, max_delay=0.05)
    rng = np.random.default_rng(2)
    reqs = [(rng.normal(size=2) * 0.1, rng.normal(size=P) * 0.1, np.array([0.5 + 0.2 * i])) for i in range(3)]

    async def go():
        out = await asyncio.gather(*[batcher(*r) for r in reqs])
        await batcher.close()
        return out

    results = asyncio.run(go())
    assert batcher.n_batches == 1
    single = GlmShards(Xs, ys, groups=[0, 1], n_groups=2, family="normal")
    for r, got in zip(reqs, results):
        want = single.reference(list(r))
        assert len(got) == 4
        for g, w in zip(got, want):
            np.testing.assert_allclose(g, w, rtol=1e-5, atol=1e-5)


def test_synth_glm_shard_draws_each_family():
    X, y, beta = synth_glm_shard(4000, P, family="negative_binomial", phi=(0.5,), seed=3, device="cpu", intercept=5.0)
    assert X.dtype == torch.bfloat16 and beta.shape == (P,)
    assert bool((y == torch.floor(y)).all()) and float(y.min()) >= 0 and float(y.max()) > 1000
    a, b, _ = synth_glm_shard(100, P, family="student_t", phi=(1.0, 3.0), seed=3, device="cpu")
    a2, b2, _ = synth_glm_shard(100, P, family="student_t", phi=(1.0, 3.0), seed=3, device="cpu")
    assert torch.equal(a, a2) and torch.equal(b, b2)
    with pytest.raises(ValueError, match="takes parameters"):
        synth_glm_shard(10, P, family="normal", phi=(), seed=0, device="cpu")


def test_negative_binomial_example_runs_on_cpu():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", B200FED_CONNECT_SLEEP="0,0")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "negative_binomial_glm.py"), "--nodes", "2",
                          "--rows", "3000", "--draws", "60"], capture_output=True, text=True, env=env, timeout=500)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "recovered" in res.stdout, res.stdout
