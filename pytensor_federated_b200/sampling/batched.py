"""Lock-step multi-chain HMC: K chains advance together, one *batched* logp/grad call per leapfrog.

This is the sampler that matches the tensor-core GLM kernels: ``GlmShards(..., n_chains=K)`` evaluates
K parameter vectors in one fused launch for (almost) the price of one, because the design matrix is
streamed from HBM once and the chains ride along the MMA's N dimension.  The reference gets chain
parallelism from one process per chain, each with its own gRPC connection
(``/root/reference/pytensor_federated/test_wrapper_ops.py:305-317``); here K chains share one launch.

``logp_dlogp_batch(theta[K, D]) -> (logp[K], grad[K, D])``.
"""
from __future__ import annotations

import dataclasses
import math
from typing import Callable, Optional, Tuple

import numpy as np

BatchFn = Callable[[np.ndarray], Tuple[np.ndarray, np.ndarray]]


@dataclasses.dataclass
class BatchedResult:
    """Draws and diagnostics of K lock-step chains (``hmc_sample_batched``)."""

    samples: np.ndarray        # [draws, K, D]
    logp: np.ndarray           # [draws, K]
    accept_rate: np.ndarray    # [K]
    step_size: np.ndarray      # [K]
    n_batched_evals: int       # number of fused launches (each evaluates K chains)
    inv_mass: Optional[np.ndarray] = None      # adapted diagonal inverse mass matrix [D]
    rng_state: Optional[dict] = None           # numpy Generator state after the last draw

    # -- checkpoint / resume, as for single chains (SamplerResult.save / .load) --------------------
    def save(self, path: str) -> None:
        import json

        np.savez(path, samples=self.samples, logp=self.logp, accept_rate=self.accept_rate, step_size=self.step_size,
                 n_batched_evals=self.n_batched_evals,
                 inv_mass=self.inv_mass if self.inv_mass is not None else np.zeros(0),
                 rng_state=np.frombuffer(json.dumps(self.rng_state, default=int).encode(), dtype=np.uint8))

    @classmethod
    def load(cls, path: str) -> "BatchedResult":
        import json

        z = np.load(path if str(path).endswith(".npz") else str(path) + ".npz")
        rng_state = json.loads(bytes(z["rng_state"]).decode()) if z["rng_state"].size else None
        return cls(samples=z["samples"], logp=z["logp"], accept_rate=z["accept_rate"], step_size=z["step_size"],
                   n_batched_evals=int(z["n_batched_evals"]), inv_mass=z["inv_mass"] if z["inv_mass"].size else None,
                   rng_state=rng_state)

    def summary(self, names=None):
        """Mean / sd / quantiles / ESS / split-R-hat per dimension over all K chains (``diagnostics.summarize``)."""
        from .diagnostics import summarize

        d = self.samples.shape[2]
        names = list(names) if names is not None else [f"theta[{i}]" for i in range(d)]
        return summarize({name: self.samples[:, :, i] for i, name in enumerate(names)})

    def rhat(self) -> np.ndarray:
        """Split-free potential scale reduction per dimension (needs K >= 2)."""
        n, k, _ = self.samples.shape
        chain_means = self.samples.mean(0)                      # [K, D]
        w = self.samples.var(0, ddof=1).mean(0)                 # within-chain
        b = n * chain_means.var(0, ddof=1)                      # between-chain
        return np.sqrt(((n - 1) / n * w + b / n) / np.maximum(w, 1e-300))


def hmc_sample_batched(logp_dlogp_batch: BatchFn, x0: np.ndarray, *, draws: int = 500, tune: int = 500,
                       n_leapfrog: int = 16, step_size: float = 0.1, target_accept: float = 0.8, seed: int = 0,
                       adapt_mass: bool = True, resume: Optional[BatchedResult] = None) -> BatchedResult:
    """Static-trajectory HMC on K chains in lock step; per-chain dual-averaging step sizes and
    diagonal mass matrices (pooled over chains).

    ``resume=<BatchedResult>`` continues finished / checkpointed chains: starts at their last draws with
    the adapted step sizes and mass matrix and the saved random state, and skips tuning — the concatenation
    of the two runs equals one longer run."""
    rng = np.random.default_rng(seed)
    if resume is not None:
        x0 = resume.samples[-1]
        tune = 0
        if resume.rng_state is not None:
            rng.bit_generator.state = resume.rng_state
    x = np.array(x0, dtype=np.float64)
    if x.ndim != 2:
        raise ValueError("x0 must be [K, D]")
    K, D = x.shape
    lp, g = logp_dlogp_batch(x)
    lp, g = np.asarray(lp, dtype=np.float64), np.asarray(g, dtype=np.float64)
    n_evals = 1
    inv_mass = np.ones(D)
    eps = np.full(K, float(step_size))
    if resume is not None:
        eps = np.array(resume.step_size, dtype=np.float64)
        if resume.inv_mass is not None:
            inv_mass = np.array(resume.inv_mass, dtype=np.float64)
    # dual averaging state per chain
    mu = np.log(10.0 * eps)
    h_bar = np.zeros(K)
    log_eps_bar = np.zeros(K)
    gamma, t0, kappa = 0.05, 10.0, 0.75
    t = 0
    samples = np.empty((draws, K, D))
    lps = np.empty((draws, K))
    acc = np.zeros(K)
    warm = []
    for it in range(tune + draws):
        p = rng.normal(size=(K, D)) / np.sqrt(inv_mass)
        h0 = lp - 0.5 * np.sum(inv_mass * p * p, axis=1)
        e = (eps * rng.uniform(0.8, 1.2, size=K))[:, None]
        xn, pn, lpn, gn = x.copy(), p.copy(), lp.copy(), g.copy()
        alive = np.ones(K, dtype=bool)
        for _ in range(n_leapfrog):
            pn = pn + 0.5 * e * gn
            xn = xn + e * inv_mass * pn
            lpn, gn = logp_dlogp_batch(xn)
            lpn, gn = np.asarray(lpn, dtype=np.float64), np.asarray(gn, dtype=np.float64)
            n_evals += 1
            bad = ~np.isfinite(lpn)
            if bad.any():  # park diverged chains on their start point so the batch stays finite
                alive &= ~bad
                xn[bad], gn[bad] = x[bad], g[bad]
                pn[bad] = 0.0
            pn = pn + 0.5 * e * gn
        h1 = np.where(alive, lpn - 0.5 * np.sum(inv_mass * pn * pn, axis=1), -np.inf)
        a = np.where(np.isfinite(h1), np.exp(np.minimum(0.0, h1 - h0)), 0.0)
        accept = rng.uniform(size=K) < a
        x[accept], lp[accept], g[accept] = xn[accept], lpn[accept], gn[accept]
        if it < tune:
            t += 1
            w = 1.0 / (t + t0)
            h_bar = (1 - w) * h_bar + w * (target_accept - a)
            log_eps = mu - math.sqrt(t) / gamma * h_bar
            eta = t ** (-kappa)
            log_eps_bar = eta * log_eps + (1 - eta) * log_eps_bar
            eps = np.exp(log_eps)
            warm.append(x.copy())
            if adapt_mass and it == int(0.6 * tune) and len(warm) > 20:
                pooled = np.asarray(warm[len(warm) // 3:]).reshape(-1, D)
                var = pooled.var(axis=0)
                inv_mass = np.where(var > 1e-12, var, 1.0)
                mu = np.log(10.0 * eps)
                h_bar[:] = 0.0
                log_eps_bar[:] = 0.0
                t = 0
            if it == tune - 1:
                eps = np.exp(log_eps_bar)
        else:
            samples[it - tune] = x
            lps[it - tune] = lp
            acc += a
    return BatchedResult(samples, lps, acc / max(1, draws), eps, n_evals, inv_mass=inv_mass,
                         rng_state=rng.bit_generator.state)


def glm_batch_fn(engine, n_groups: int) -> BatchFn:
    """Adapts a multi-chain ``FederatedEngine(GlmShards(..., n_chains=K))`` to the batched signature
    with ``theta = [intercept[G], beta[P]]`` per chain (flat prior; add priors by wrapping).

    For the families with fitted parameters phi (``normal``, ``student_t``, ``negative_binomial``) the sampler
    works on the unconstrained ``theta = [intercept[G], beta[P], log phi[D]]``: phi = exp(theta[G+P:]), the
    gradient is taken through the chain rule and the log-Jacobian ``sum(log phi)`` is added to logp, so a flat
    prior on log phi is the improper prior ``1 / phi`` on phi.

    Any number of chains may be passed: the kernel's capacity per launch is ``K`` (at most 16 for the bf16
    tensor-core kernel, 3 for the fp8 kernel); more chains are evaluated in ``ceil(chains / K)`` launches and a
    short last tile is padded by repeating its last chain, so 64 chains on a K = 16 engine cost four passes over the
    data instead of sixty-four."""
    cap = int(getattr(engine.model, "n_chains", 1))
    D = int(getattr(engine.model, "n_family_params", 0))

    def evaluate(theta: np.ndarray):
        """theta ``[cap, G+P(+D)]`` -> (logp ``[cap]``, grad ``[cap, G+P(+D)]``) in the sampler's coordinates."""
        single = cap == 1   # single-chain engines take unbatched inputs
        rows = theta[0] if single else theta
        G = n_groups
        if not D:
            logp, d_ic, d_beta = engine.evaluate(rows[..., :G], rows[..., G:])
            return np.asarray(logp).reshape(-1), np.concatenate(
                [np.asarray(d_ic).reshape(cap, -1), np.asarray(d_beta).reshape(cap, -1)], axis=1)
        log_phi = rows[..., -D:]
        phi = np.exp(log_phi)
        logp, d_ic, d_beta, d_phi = engine.evaluate(rows[..., :G], rows[..., G:-D], phi)
        logp = np.asarray(logp).reshape(-1) + np.asarray(log_phi).reshape(cap, D).sum(axis=1)
        d_log_phi = np.asarray(d_phi).reshape(cap, D) * phi.reshape(cap, D) + 1.0
        return logp, np.concatenate([np.asarray(d_ic).reshape(cap, -1), np.asarray(d_beta).reshape(cap, -1), d_log_phi], axis=1)

    def fn(theta: np.ndarray):
        theta = np.asarray(theta)
        n = theta.shape[0]
        if n == cap and cap > 1:
            return evaluate(theta)
        logps, grads = [], []
        for first in range(0, n, cap):
            block = theta[first : first + cap]
            k = block.shape[0]
            if k < cap:
                block = np.concatenate([block, np.repeat(block[-1:], cap - k, axis=0)], axis=0)
            lp, gr = evaluate(block)
            logps.append(lp[:k])
            grads.append(gr[:k])
        return np.concatenate(logps), np.concatenate(grads, axis=0)

    return fn


__all__ = ["BatchedResult", "hmc_sample_batched", "glm_batch_fn"]
