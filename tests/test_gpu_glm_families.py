"""Families with fitted parameters on the tensor-core GLM kernel vs the fp64 oracle (needs a B200; the world-2
case needs two)."""
import os
import socket

import numpy as np
import pytest
import torch

from pytensor_federated_b200.models import GlmShards, synth_glm_shard
from pytensor_federated_b200.parallel import FederatedEngine

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

FAMILIES = ["normal", "student_t", "negative_binomial"]
DATA_PHI = {"normal": (0.7,), "student_t": (1.3, 4.0), "negative_binomial": (2.0,)}
EVAL_PHI = {"normal": [0.8], "student_t": [1.2, 4.5], "negative_binomial": [2.5]}
ROWS = [128 * 37, 77, 4099, 128, 1]          # whole tiles, a sub-tile segment, a 1-row segment
GROUPS = [0, 1, 0, 2, 1]


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pytensor_federated_b200.ops import native

    native.load()  # a GPU box without the native library is a failure, not a skip
    return torch.device("cuda:0")


def _case(dev, family, rows, P, seed=0, intercept=0.5, phi=None):
    Xs, ys = [], []
    for i, n in enumerate(rows):
        X, y, _ = synth_glm_shard(n, P, family=family, phi=phi or DATA_PHI.get(family, ()), seed=seed + i, device=dev,
                                  beta_scale=0.05, intercept=intercept)
        Xs.append(X)
        ys.append(y)
    return Xs, ys


def _params(K, P, family, seed=2):
    rng = np.random.default_rng(seed)
    base = np.asarray(EVAL_PHI[family])
    if K == 1:
        return np.array([0.3, -0.2, 0.1]), (rng.normal(size=P) * 0.03).astype(np.float32), base
    ic = rng.normal(size=(K, 3)) * 0.2
    beta = (rng.normal(size=(K, P)) * 0.03).astype(np.float32)
    phi = base[None, :] * np.exp(rng.normal(size=(K, base.size)) * 0.3)
    return ic, beta, phi.astype(np.float32)


def _check(got, want, n_rows):
    logp, d_ic, d_beta, d_phi = got
    w_logp, w_ic, w_beta, w_phi = want
    np.testing.assert_allclose(logp, w_logp, rtol=2e-5)
    np.testing.assert_allclose(d_ic, w_ic, rtol=1e-4, atol=2e-3)
    np.testing.assert_allclose(d_beta, w_beta, rtol=1e-4, atol=2e-3 * np.sqrt(n_rows))
    np.testing.assert_allclose(d_phi, w_phi, rtol=1e-4, atol=2e-3 * np.sqrt(n_rows))


@pytest.mark.parametrize("P", [256, 72, 384])
@pytest.mark.parametrize("family", FAMILIES)
def test_tensor_core_matches_oracle(dev, family, P):
    Xs, ys = _case(dev, family, ROWS, P)
    model = GlmShards(Xs, ys, groups=GROUPS, n_groups=3, family=family, kernel="tc")
    ic, beta, phi = _params(1, P, family)
    with FederatedEngine(model) as eng:
        assert model.selected_kernel == "tc"
        got = eng.evaluate(ic, beta, phi)
        again = eng.evaluate(ic, beta, phi)
    assert got[3].shape == (len(phi),)
    want = model.unpack_result(model.reference_partial([ic, beta, phi], dtype=torch.float64))
    _check(got, want, sum(ROWS))
    for u, v in zip(got, again):
        assert np.array_equal(u, v), "two evaluations of the same theta must agree bit for bit"


@pytest.mark.parametrize("K", [4, 8, 16])
@pytest.mark.parametrize("family", FAMILIES)
def test_tensor_core_batches_chains(dev, family, K):
    rows = [128 * 50 + 5, 3000, 1]
    Xs, ys = _case(dev, family, rows, 256, seed=9)
    model = GlmShards(Xs, ys, groups=[0, 1, 2], n_groups=3, family=family, n_chains=K, kernel="tc")
    ic, beta, phi = _params(K, 256, family)
    with FederatedEngine(model) as eng:
        got = eng.evaluate(ic, beta, phi)
        again = eng.evaluate(ic, beta, phi)
    assert got[0].shape == (K,) and got[3].shape == (K, phi.shape[1])
    want = model.unpack_result(model.reference_partial([ic, beta, phi], dtype=torch.float64))
    _check(got, want, sum(rows))
    for u, v in zip(got, again):
        assert np.array_equal(u, v)


@pytest.mark.parametrize("family", FAMILIES)
def test_per_node_output_blocks(dev, family):
    rows = [128 * 20 + 3, 900, 128 * 9, 1]
    Xs, ys = _case(dev, family, rows, 128, seed=4)
    K = 4
    model = GlmShards(Xs, ys, groups=[0, 1, 2, 0], n_groups=3, family=family, n_chains=K, kernel="tc",
                      node_ids=[0, 1, 2, 1], n_nodes=3)
    ic, beta, phi = _params(K, 128, family, seed=6)
    with FederatedEngine(model) as eng:
        per = model.per_node(eng.evaluate_raw([ic, beta, phi]))
    want = model.per_node(model.reference_partial([ic, beta, phi], dtype=torch.float64))
    assert per.shape == (3, K, 1 + 3 + 128 + len(EVAL_PHI[family]))
    for node in range(3):
        n_rows = sum(r for r, i in zip(rows, [0, 1, 2, 1]) if i == node)
        np.testing.assert_allclose(per[node, :, 0], want[node, :, 0], rtol=2e-5)
        np.testing.assert_allclose(per[node, :, 1:], want[node, :, 1:], rtol=1e-4, atol=2e-3 * np.sqrt(n_rows))


@pytest.mark.parametrize("alpha", [0.5, 5.0, 500.0])
@pytest.mark.parametrize("K", [1, 16])
def test_negative_binomial_dispersions_and_large_counts(dev, alpha, K):
    # overdispersed counts around mu ~ exp(5): many above the short-sum cutoff, some above 1000
    rows = [128 * 60 + 11, 2000]
    Xs, ys = _case(dev, "negative_binomial", rows, 256, seed=13, intercept=5.0, phi=(0.5,))
    assert max(float(y.max()) for y in ys) > 1000
    model = GlmShards(Xs, ys, groups=[0, 1], n_groups=2, family="negative_binomial", n_chains=K, kernel="tc")
    rng = np.random.default_rng(3)
    if K == 1:
        ic, beta, phi = np.array([5.0, 4.9]), (rng.normal(size=256) * 0.03).astype(np.float32), np.array([alpha])
    else:
        ic = 5.0 + rng.normal(size=(K, 2)) * 0.1
        beta = (rng.normal(size=(K, 256)) * 0.03).astype(np.float32)
        phi = (alpha * np.exp(rng.normal(size=(K, 1)) * 0.2)).astype(np.float32)
    with FederatedEngine(model) as eng:
        got = eng.evaluate(ic, beta, phi)
        again = eng.evaluate(ic, beta, phi)
    want = model.unpack_result(model.reference_partial([ic, beta, phi], dtype=torch.float64))
    _check(got, want, sum(rows))
    for u, v in zip(got, again):
        assert np.array_equal(u, v)


def test_existing_families_and_new_ones_share_an_engine_process(dev):
    """A logistic engine next to a negative-binomial one: each launches its own kernel variant."""
    Xs, ys = _case(dev, "negative_binomial", [5000], 256)
    Xl, yl = _case(dev, "logistic", [5000], 256)
    nb = GlmShards(Xs, ys, family="negative_binomial", kernel="tc")
    lg = GlmShards(Xl, yl, kernel="tc")
    beta = np.zeros(256, np.float32)
    with FederatedEngine(nb) as a, FederatedEngine(lg) as b:
        r_nb = a.evaluate(np.array([0.5]), beta, np.array([2.0]))
        r_lg = b.evaluate(np.array([0.5]), beta)
    assert len(r_nb) == 4 and len(r_lg) == 3
    np.testing.assert_allclose(r_lg[0], lg.reference([np.array([0.5]), beta])[0], rtol=2e-5)


# ------------------------------------------------------------------ world 2: fused multi-GPU path
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        X, y, _ = synth_glm_shard(30_000 + 17 * rank, 256, family="negative_binomial", phi=(1.5,), seed=50 + rank,
                                  device=dev, intercept=2.0)
        K = 4
        model = GlmShards([X], [y], groups=[rank % 2], n_groups=2, family="negative_binomial", n_chains=K, kernel="tc")
        eng = FederatedEngine(model, timeout=20.0)
        rng = np.random.default_rng(1)
        ic = 2.0 + rng.normal(size=(K, 2)) * 0.1
        beta = (rng.normal(size=(K, 256)) * 0.03).astype(np.float32)
        phi = np.array([[0.5], [1.5], [5.0], [500.0]], dtype=np.float32)
        local = model.reference_partial([ic, beta, phi], dtype=torch.float64)
        gathered = [None] * world
        dist.all_gather_object(gathered, local)
        if rank == 0:
            got = eng.evaluate(ic, beta, phi)
            again = eng.evaluate(ic, beta, phi)
            same = all(np.array_equal(a, b) for a, b in zip(got, again))
            want = model.unpack_result(np.sum(gathered, axis=0), model.call_context([ic, beta, phi]))
            q.put(("root", [np.asarray(g).tolist() for g in got], [np.asarray(w).tolist() for w in want], same,
                   sum(int(n) for n in [30_000, 30_017])))
            eng.shutdown()
        else:
            eng.serve()
            eng.shutdown()
            q.put(("peer",))
    finally:
        dist.destroy_process_group()


@pytest.mark.multigpu
def test_negative_binomial_across_two_gpus_matches_gathered_oracle():
    import torch.multiprocessing as mp

    world = 2
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    root = [r for r in results if r[0] == "root"][0]
    got, want, same, n_rows = root[1], root[2], root[3], root[4]
    assert same, "two evaluations of the same theta must agree bit for bit"
    _check([np.asarray(g) for g in got], [np.asarray(w) for w in want], n_rows)
