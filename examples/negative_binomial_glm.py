"""Overdispersed count regression on federated nodes: a negative-binomial GLM whose dispersion alpha is inferred
with the coefficients (GPUs, or CPU processes for a dry run):

    python examples/negative_binomial_glm.py --nodes 4 --draws 300

Every node holds private counts ``y ~ NegativeBinomial(mu = exp(intercept + X beta), alpha)`` (PyMC's NB2
parameterisation, ``var = mu + mu^2 / alpha``).  The model is the one a PyMC user would write —

    alpha = m.HalfNormal("alpha", 5)
    beta = m.Normal("beta", 0, 1, size=P)
    for op in fed.node_ops(): m.Potential(..., op(intercept, beta, alpha)[0])

— and NUTS samples it.  Each node's term is a ``FederatedLogpGradOp``; the ``fuse_asyncs`` rewrite answers all of
them with ONE fused launch per model evaluation, and on the GPU the log-likelihood and the gradients for the
intercept, beta AND alpha come out of the same single pass of the tensor-core kernel over X.
"""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

ALPHA, INTERCEPT = 2.0, 1.0


def true_beta(P: int) -> np.ndarray:
    return np.random.default_rng(7).normal(size=P).astype(np.float32) * 0.3


class Counts:
    """Picklable model factory: node r of `world` holds the nodes r, r + world, ... (private counts of each)."""

    def __init__(self, n: int, rows: int, P: int) -> None:
        self.n, self.rows, self.P = n, rows, P

    def __call__(self, rank: int, world: int, device):
        from pytensor_federated_b200.models import GlmShards, synth_glm_shard

        mine = [s for s in range(self.n) if s % world == rank]
        Xs, ys = [], []
        for s in mine:
            X, y, _ = synth_glm_shard(self.rows + 17 * s, self.P, family="negative_binomial", phi=(ALPHA,), seed=100 + s,
                                      device=device, intercept=INTERCEPT, beta_true=true_beta(self.P))
            Xs.append(X)
            ys.append(y)
        return GlmShards(Xs, ys, family="negative_binomial", node_ids=mine, n_nodes=self.n,
                         kernel="auto" if device.type == "cuda" else "simt")


def build(fed, P: int):
    from pytensor_federated_b200.sampling import Model

    m = Model()
    intercept = m.Normal("intercept", 0.0, 5.0)
    beta = m.Normal("beta", 0.0, 1.0, size=P)
    alpha = m.HalfNormal("alpha", 5.0)
    for i, op in enumerate(fed.node_ops()):
        logp, *_ = op(intercept, beta, alpha)
        m.Potential(f"counts_{i}", logp)
    m.compile()
    return m


def main():
    import torch

    from pytensor_federated_b200.federation import NodeFederation, launch_federation
    from pytensor_federated_b200.sampling import nuts_sample

    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=4)
    ap.add_argument("--gpus", type=int, default=0, help="processes / GPUs to spread the nodes over (0 = all visible, or 1 on CPU)")
    ap.add_argument("--rows", type=int, default=20_000, help="rows per node")
    ap.add_argument("--features", type=int, default=8)
    ap.add_argument("--draws", type=int, default=200)
    args = ap.parse_args()

    visible = torch.cuda.device_count() if torch.cuda.is_available() else 0
    world = max(1, min(args.nodes, args.gpus or visible or 1))
    P = args.features
    with launch_federation(Counts(args.nodes, args.rows, P), world, device_type="cuda" if visible else "cpu",
                           backend="auto" if visible else "collective") as engine:
        fed = NodeFederation(engine)
        print(f"{args.nodes} nodes x ~{args.rows} counts on {world} {'GPU(s)' if visible else 'CPU process(es)'}, "
              f"backend={engine.backend}")
        m = build(fed, P)
        fed.n_launches = 0
        t0 = time.perf_counter()

        def logp_dlogp(theta):
            # the step-size search can propose log(alpha) so negative that alpha underflows to 0, which the model
            # rejects (phi must be > 0): to the sampler that is a proposal of zero density
            try:
                return m.logp_dlogp(theta)
            except ValueError:
                return -np.inf, np.zeros_like(theta)

        res = nuts_sample(logp_dlogp, np.zeros(m.dim), draws=args.draws, tune=args.draws, seed=5)
        dt = time.perf_counter() - t0
        post = m.point(res.samples.mean(0))
        alpha, beta = float(post["alpha"]), np.asarray(post["beta"])
        err = float(np.abs(beta - true_beta(P)).max())
        print(f"NUTS: {res.n_logp_evals} model evaluations = {fed.n_launches} fused launches in {dt:.2f} s")
        print(f"alpha = {alpha:.2f} (true {ALPHA}), intercept = {float(post['intercept']):.2f} (true {INTERCEPT}), "
              f"max |beta - beta_true| = {err:.3f}")
        ok = abs(alpha - ALPHA) < 0.3 * ALPHA and abs(float(post["intercept"]) - INTERCEPT) < 0.2 and err < 0.1
        print("recovered alpha and beta" if ok else "NOT recovered")
        if not ok:
            sys.exit(1)


if __name__ == "__main__":
    main()
